"""Formation-family kernels (csrc/fm_formation.cu through fm_formation_*) against the float64 oracle
(oracle/formation.py, itself pinned to the unmodified reference by tests/test_oracle_formation.py)."""
from dataclasses import fields

import numpy as np
import pytest

from oracle.formation import FormationConfig, FormationOracle, FormationState
from oracle.make_formation_golden import load, set_walls, state_from
from oracle.navgraph import INFO_KEYS
from parity_util import assert_close, assert_fairness_close

pytestmark = pytest.mark.gpu

INT_FIELDS = ("goal_match", "step", "episode")
RATIO_KEYS = ("Mean_by_variance", "Time_mean_by_stddev")


def _sim(cfg: FormationConfig, **kw):
    from fair_marl_b200 import FormationSimConfig
    return FormationSimConfig(
        num_agents=cfg.num_agents, num_obstacles=cfg.num_obstacles, world_size=cfg.world_size, max_speed=cfg.max_speed,
        collision_rew=cfg.collision_rew, goal_rew=cfg.goal_rew, min_dist_thresh=cfg.min_dist_thresh,
        min_obs_dist=cfg.min_obs_dist, episode_length=cfg.episode_length, fair_rew=cfg.fair_rew, zeroshift=cfg.zeroshift,
        collaborative=cfg.collaborative, fairness_reward=cfg.fairness_reward, assignment=cfg.assignment,
        num_walls=cfg.num_walls, **kw)


def _fp32(st: FormationState) -> FormationState:
    d = {}
    for f in fields(FormationState):
        a = np.asarray(getattr(st, f.name))
        if f.name in INT_FIELDS:
            d[f.name] = a.astype(np.int64)
        elif f.name == "status":
            d[f.name] = a.astype(bool)
        else:
            with np.errstate(over="ignore"):
                d[f.name] = a.astype(np.float32).astype(np.float64)
    return FormationState(**d)


def _to_device(st: FormationState):
    return {f.name: (np.asarray(getattr(st, f.name)).astype(np.uint8) if f.name == "status" else np.asarray(getattr(st, f.name)))
            for f in fields(FormationState)}


def _from_device(dev) -> FormationState:
    d = {}
    for f in fields(FormationState):
        a = dev[f.name].cpu().numpy()
        d[f.name] = a.astype(np.int64) if f.name in INT_FIELDS else (a.astype(bool) if f.name == "status" else a.astype(np.float64))
    return FormationState(**d)


def _walls_to_device(orc: FormationOracle):
    """Wall geometry of the oracle (kept beside FormationState) as device state entries, rounded to fp32 like the rest."""
    if not orc.cfg.num_walls:
        return {}
    return {"wall_axis": orc.wall_axis.astype(np.float32), "wall_orient": orc.wall_orient.astype(np.int32),
            "wall_len": orc.wall_len.astype(np.float32)}


def _walls_from_device(orc: FormationOracle, dev) -> None:
    if orc.cfg.num_walls:
        orc.wall_axis = dev["wall_axis"].cpu().numpy().astype(np.float64)
        orc.wall_orient = dev["wall_orient"].cpu().numpy().astype(np.int64)
        orc.wall_len = dev["wall_len"].cpu().numpy().astype(np.float64)


def _np(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


def _actions(a):
    import torch
    return torch.as_tensor(np.asarray(a), dtype=torch.int32, device="cuda")


def _compare_step(out, ref, post: FormationState, rpost: FormationState):
    assert_close(out["obs"], ref["obs"], "obs")
    assert_close(out["node_obs"], ref["node_obs"], "node_obs")
    assert_close(out["adj_env"], ref["adj"], "adj")
    assert_close(out["reward"], ref["reward"], "reward")
    assert (out["done"].astype(bool) == ref["done"]).all(), "done"
    for k, key in enumerate(INFO_KEYS):
        (assert_fairness_close if key in RATIO_KEYS else assert_close)(out["info"][..., k], ref["info"][key], key)
    for f in ("goal_match", "step", "status"):
        assert (getattr(post, f) == getattr(rpost, f)).all(), f


@pytest.mark.parametrize("name", ["formation_n3_o3_fafr", "formation_n4_o2_fa", "formation_n7_o3_fafr", "formation_n3_o3_oa",
                                  "formation_n3_o3_ra", "formation_n3_o2_w2", "formation_n3_o3_w1_oa"])
def test_step_matches_oracle_on_reference_states(name):
    """One step from every recorded reference state (rounded to fp32): device vs float64 oracle, outputs, info and the
    whole post-step state -- status latches, occupancy table, goal history and nearest-landmark latches included."""
    import fair_marl_b200 as fm
    cfg, g = load(name)
    pre = _fp32(state_from(g, "pre_"))
    T = pre.pos.shape[0]
    env = fm.B200FormationVecEnv(_sim(cfg, auto_reset=False), num_envs=T)
    orc = FormationOracle(cfg, T)
    orc.set_state(pre)
    set_walls(orc, g, "pre_")
    dev_walls = _walls_to_device(orc)
    env.set_state({**_to_device(pre), **dev_walls})
    _walls_from_device(orc, env.get_state())                  # the fp32 geometry the device holds
    out = _np(env.step_tensor(_actions(g["actions"])))
    ref = orc.step(g["actions"], autoreset=False)
    post, rpost = _from_device(env.get_state()), orc.get_state()
    _compare_step(out, ref, post, rpost)
    for f in ("pos", "vel", "p_dist", "dists_to_goal", "times_required", "dist_left_to_goal", "num_agent_collisions",
              "num_obstacle_collisions", "dist_traveled_mean", "dist_traveled_stddev", "goal_reached", "occupied", "goal_history"):
        assert_close(getattr(post, f), getattr(rpost, f), f)
    # smooth quantities straight against the reference's own float64 outputs (inputs were rounded to fp32 on the way in)
    assert_close(out["adj_env"], g["out_adj"], "adj vs reference")
    assert_close(out["obs"][..., :4], g["out_obs"][..., :4], "vel / pos vs reference")
    assert orc.branch_hits.get("status_latched", 0) > 0
    if cfg.assignment == "fair":
        assert orc.branch_hits.get("subset_index_quirk", 0) > 0
    if cfg.num_walls:
        assert orc.branch_hits.get("wall_end_cap", 0) > 0 and orc.branch_hits.get("wall_box_hit", 0) > 0
        assert (out["node_obs"][:, :, -cfg.num_walls:, 12] == 3.0).all()
    env.close()


def _goal_seeking(st: FormationState, rng) -> np.ndarray:
    """Actions [B,N]: the move along the larger axis of (assigned goal - position), a random move with probability 1/4."""
    B, N = st.goal_match.shape
    d = np.take_along_axis(st.landmark_pos, st.goal_match[..., None], axis=1) - st.pos
    seek = np.where(np.abs(d[..., 0]) > np.abs(d[..., 1]), np.where(d[..., 0] > 0, 1, 2), np.where(d[..., 1] > 0, 3, 4))
    return np.where(rng.random((B, N)) < 0.25, rng.integers(0, 5, (B, N)), seek)


# The step kernels of the formation family: steps with N <= 4, O <= 3 and no walls run the split path
# (formation_logic_kernel<N, O> + formation_image_kernel<N, O>, one instantiation per pair of this grid); FM_FORM_FUSED=1
# sends them to formation_kernel<N, 0, -1>, which every other shape (N >= 5, O >= 4, walls) takes anyway.
SPLIT_GRID = [(N, O) for N in (2, 3, 4) for O in (0, 1, 2, 3)]
SHORT = dict(episode_length=12, steps=30)          # two or three episodes per env: time-outs inside the rollout


def _case(N, O, B, collab, fair, assignment, W, tag="", **opts):
    """One reset + rollout case.  opts: fused (FM_FORM_FUSED=1), max_speed, episode_length, steps, early (at least one env
    must finish early, every agent latched).  The id is pytest's own for the first seven values, plus the tag."""
    ident = "-".join(str(v) for v in (N, O, B, collab, fair, assignment, W)) + (f"-{tag}" if tag else "")
    return pytest.param(N, O, B, collab, fair, assignment, W, opts, id=ident)


ORACLE_CASES = [
    _case(3, 3, 48, False, True, "fair", 0, early=True), _case(4, 2, 32, True, False, "fair", 0, early=True),
    _case(2, 1, 32, False, True, "fair", 0, early=True),
    _case(3, 3, 70, False, True, "fair", 0, early=True),                # a ragged last warp: the lane-store emission path
    _case(5, 2, 32, False, True, "fair", 0), _case(7, 3, 40, False, True, "fair", 0),   # N > 4: serial lexifair descent every step
    _case(3, 3, 48, False, False, "optimal", 0, early=True), _case(4, 1, 32, True, False, "optimal", 0, early=True),
    _case(3, 3, 48, False, False, "random", 0, early=True), _case(6, 2, 32, False, False, "random", 0),
    _case(3, 2, 40, False, True, "fair", 2, early=True), _case(4, 3, 32, False, False, "optimal", 1, early=True),   # walls
    _case(5, 1, 32, False, True, "fair", 2),
    # every split instantiation, ragged batches (B = 1 and below the image kernel's 16-env CTA included), short episodes
    _case(2, 0, 1, False, True, "fair", 0, **SHORT), _case(2, 1, 17, True, False, "optimal", 0, **SHORT, early=True),
    _case(2, 2, 37, False, False, "random", 0, **SHORT, early=True), _case(2, 3, 45, False, True, "fair", 0, **SHORT, early=True),
    _case(3, 0, 17, False, False, "optimal", 0, **SHORT), _case(3, 1, 45, True, True, "fair", 0, **SHORT),
    _case(3, 2, 37, False, False, "fair", 0, **SHORT, early=True), _case(3, 3, 1, False, False, "random", 0, **SHORT),
    _case(4, 0, 45, False, False, "random", 0, **SHORT), _case(4, 1, 37, False, True, "fair", 0, **SHORT),
    _case(4, 2, 17, True, False, "optimal", 0, **SHORT), _case(4, 3, 45, False, False, "fair", 0, **SHORT),
    # the same twelve shapes on the fused kernel
    _case(2, 0, 45, False, False, "optimal", 0, "fused", fused=True, **SHORT, early=True),
    _case(2, 1, 37, False, True, "fair", 0, "fused", fused=True, **SHORT, early=True),
    _case(2, 2, 1, True, False, "fair", 0, "fused", fused=True, **SHORT),
    _case(2, 3, 17, False, False, "random", 0, "fused", fused=True, **SHORT, early=True),
    _case(3, 0, 45, True, True, "fair", 0, "fused", fused=True, **SHORT),
    _case(3, 1, 17, False, False, "random", 0, "fused", fused=True, **SHORT),
    _case(3, 2, 45, False, False, "optimal", 0, "fused", fused=True, **SHORT, early=True),
    _case(3, 3, 37, False, True, "fair", 0, "fused", fused=True, **SHORT),
    _case(4, 0, 17, False, True, "fair", 0, "fused", fused=True, **SHORT),
    _case(4, 1, 1, False, False, "optimal", 0, "fused", fused=True, **SHORT),
    _case(4, 2, 45, False, False, "random", 0, "fused", fused=True, **SHORT),
    _case(4, 3, 37, True, False, "fair", 0, "fused", fused=True, **SHORT),
    # large obstacle counts (fused kernel; O = 8 is FM_FORMATION_MAX_OBSTACLES, E up to 24)
    _case(2, 8, 37, False, True, "fair", 0, **SHORT, early=True), _case(4, 4, 45, False, False, "optimal", 0, **SHORT),
    _case(5, 6, 17, False, False, "random", 0, **SHORT), _case(7, 8, 17, False, True, "fair", 0, **SHORT),
    _case(7, 8, 17, False, False, "fair", 2, **SHORT), _case(4, 8, 33, True, False, "optimal", 1, **SHORT),
    # no max_speed (min_time is never written; the pending reset keeps it too) and a max_speed that clips often
    _case(3, 2, 37, False, True, "fair", 0, "vmax_none", max_speed=None, **SHORT, early=True),
    _case(3, 2, 37, False, True, "fair", 0, "vmax_0.7", max_speed=0.7, **SHORT, early=True),
    _case(5, 3, 17, False, False, "optimal", 0, "vmax_none", max_speed=None, **SHORT),
    _case(5, 3, 17, False, False, "optimal", 0, "vmax_0.7", max_speed=0.7, **SHORT),
]


def test_oracle_cases_cover_the_split_grid():
    """Every (N, O) instantiation of the split step path is stepped against the oracle, on the split kernels and on the fused
    kernel: trimming the list above must not silently drop one."""
    split, fused = set(), set()
    for case in ORACLE_CASES:
        N, O, B, collab, fair, assignment, W, opts = case.values
        if W == 0 and (N, O) in SPLIT_GRID:
            (fused if opts.get("fused") else split).add((N, O))
    assert split == set(SPLIT_GRID), sorted(set(SPLIT_GRID) - split)
    assert fused == set(SPLIT_GRID), sorted(set(SPLIT_GRID) - fused)


@pytest.mark.parametrize("N,O,B,collab,fair,assignment,W,opts", ORACLE_CASES)
def test_reset_and_rollout_match_oracle(N, O, B, collab, fair, assignment, W, opts, monkeypatch):
    """Device reset == oracle reset bit for bit (same Philox draws, same acceptance rules, same lexifair), then a rollout
    that steers at the goals (so agents latch and envs finish early) across auto-resets, compared step by step."""
    if opts.get("fused"):
        monkeypatch.setenv("FM_FORM_FUSED", "1")
    cfg = FormationConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0,
                          episode_length=opts.get("episode_length", 15), max_speed=opts.get("max_speed", 2.0),
                          collaborative=collab, fairness_reward=fair, assignment=assignment, num_walls=W)
    _rollout_matches_oracle(cfg, B, opts.get("steps", 32), opts.get("early", False))


def _rollout_matches_oracle(cfg: FormationConfig, B: int, steps: int, early: bool):
    import fair_marl_b200 as fm
    W = cfg.num_walls
    env = fm.B200FormationVecEnv(_sim(cfg), num_envs=B, seed=7, env_offset=3)
    orc = FormationOracle(cfg, B, seed=7, env_offset=3)
    if cfg.max_speed is None:                     # a reset leaves min_time alone then: start from the device's zeroed block
        orc.s.min_time[:] = 0.0
    out, ref = _np(env.reset_tensor()), orc.reset()
    st, rs = _from_device(env.get_state()), orc.get_state()
    if W:                                         # same draws, same fp32 arithmetic: the wall geometry is bit-identical
        dev = env.get_state()
        assert (dev["wall_axis"].cpu().numpy() == orc.wall_axis.astype(np.float32)).all()
        assert (dev["wall_orient"].cpu().numpy() == orc.wall_orient).all()
        assert (dev["wall_len"].cpu().numpy() == orc.wall_len.astype(np.float32)).all()
    for f in ("pos", "landmark_pos", "obstacle_pos"):
        assert (getattr(st, f) == getattr(rs, f)).all(), f
    assert (st.goal_match == rs.goal_match).all() and (st.episode == 1).all() and not st.status.any()
    assert_close(st.min_time, rs.min_time, "min_time")
    assert_close(st.occupied, rs.occupied, "occupancy after the reset observation")
    assert_close(out["obs"], ref["obs"], "reset obs")
    assert_close(out["node_obs"], ref["node_obs"], "reset node_obs")
    assert_close(out["adj_env"], ref["adj"], "reset adj")
    rng = np.random.default_rng(5)
    resets = early_resets = 0
    for t in range(steps):
        dev = env.get_state()
        cur = _from_device(dev)
        orc.set_state(cur)
        _walls_from_device(orc, dev)
        a = _goal_seeking(cur, rng)
        out = _np(env.step_tensor(_actions(a)))
        ref = orc.step(a, autoreset=True)
        post, rpost = _from_device(env.get_state()), orc.get_state()
        _compare_step(out, ref, post, rpost)
        hit = ref["reset"]
        resets += int(hit.sum())
        early_resets += int((hit & (cur.step + 1 < cfg.episode_length)).sum())
        assert (post.episode == rpost.episode).all()
        if hit.any():
            assert (post.pos[hit] == rpost.pos[hit]).all() and (post.landmark_pos[hit] == rpost.landmark_pos[hit]).all()
            assert (post.obstacle_pos[hit] == rpost.obstacle_pos[hit]).all()
            assert (post.goal_match[hit] == rpost.goal_match[hit]).all()
            if W:
                dev = env.get_state()
                assert (dev["wall_axis"].cpu().numpy()[hit] == orc.wall_axis[hit].astype(np.float32)).all()
                assert (dev["wall_orient"].cpu().numpy()[hit] == orc.wall_orient[hit]).all()
                assert (dev["wall_len"].cpu().numpy()[hit] == orc.wall_len[hit].astype(np.float32)).all()
        assert_close(post.pos, rpost.pos, "pos")
        assert_close(post.min_time, rpost.min_time, "min_time")
        assert_close(post.occupied, rpost.occupied, "occupied")
        assert_close(post.goal_history, rpost.goal_history, "goal_history")
    assert resets >= B                            # time-outs ...
    if early:
        assert early_resets > 0                   # ... and all-agents-latched early resets both happened
    env.close()


@pytest.mark.parametrize("N,O,B,T,slots", [(3, 3, 4096 + 70, 40, 40), (4, 2, 8192, 12, 12), (3, 3, 300, 30, 4), (5, 2, 4500, 9, 9)])
@pytest.mark.parametrize("lanes", ["1", "2"])
def test_rollout_lanes_equal_single_steps(N, O, B, T, slots, lanes, monkeypatch):
    """fm_formation_step_many (one lane, or two env-range lanes on two streams for B >= 4096; pre-generated actions) against T calls of
    fm_formation_step: every output of every step still in the ring, the final state and the info rows, bit for bit.
    Short episodes, so that time-out resets fall inside the rollout; goal seeking, so that early resets do too."""
    import torch
    import fair_marl_b200 as fm
    monkeypatch.setenv("FM_FORM_LANES", lanes)
    cfg = FormationConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=7)
    e_r = fm.B200FormationVecEnv(_sim(cfg, info_every_step=False), num_envs=B, seed=11, num_slots=slots)
    e_s = fm.B200FormationVecEnv(_sim(cfg, info_every_step=False), num_envs=B, seed=11, num_slots=slots)
    e_r.reset_tensor(); e_s.reset_tensor()
    g = torch.Generator(device="cuda").manual_seed(5)
    acts = torch.randint(0, 5, (T, B, N), generator=g, device="cuda", dtype=torch.int32)
    slot_of = e_r.rollout_tensor(acts)
    for t in range(T):
        o_s = e_s.step_tensor(acts[t])
        if slot_of[t] not in slot_of[t + 1:]:
            o_r = e_r.slot_outputs(slot_of[t])
            for k in ("obs", "node_obs", "adj_env", "reward", "done"):
                assert torch.equal(o_r[k], o_s[k]), (t, k)
    s_r, s_s = e_r.get_state(), e_s.get_state()
    for k in s_r:
        assert torch.equal(s_r[k], s_s[k]), k
    assert torch.equal(e_r._slots[0]["info"], e_s._slots[0]["info"])
    assert int(s_r["episode"].max()) >= 1 + T // 7
    # a second rollout continues the same trajectory
    slot_of = e_r.rollout_tensor(acts[:3])
    for t in range(3):
        o_s = e_s.step_tensor(acts[t])
        assert torch.equal(e_r.slot_outputs(slot_of[t])["node_obs"], o_s["node_obs"]), t
    e_r.close(); e_s.close()


def test_masked_reset_and_errors():
    import torch
    import fair_marl_b200 as fm
    cfg = FormationConfig(num_agents=3, num_obstacles=2)
    env = fm.B200FormationVecEnv(_sim(cfg), num_envs=40, seed=1)
    env.reset_tensor()
    before = _from_device(env.get_state())
    mask = np.zeros(40, np.uint8); mask[::3] = 1
    env.reset_tensor(mask)
    after = _from_device(env.get_state())
    keep = mask == 0
    assert (after.pos[keep] == before.pos[keep]).all() and (after.episode[keep] == 1).all()
    assert (after.episode[~keep] == 2).all() and (after.pos[~keep] != before.pos[~keep]).any()
    with pytest.raises(ValueError):
        env.step_tensor(torch.zeros((40, 3), dtype=torch.int64, device="cuda"))
    with pytest.raises(fm._lib.FairMarlError):
        fm.B200FormationVecEnv(fm.FormationSimConfig(num_agents=8), num_envs=8)
    with pytest.raises(fm._lib.FairMarlError):                          # the base scenarios have no fairness term
        fm.B200FormationVecEnv(fm.FormationSimConfig(assignment="optimal", fairness_reward=True), num_envs=8)
    env.close()


def test_info_rows_only_when_every_agent_is_done():
    """info_every_step = False (rollouts): the info rows are written on the steps on which every agent of the env is done
    -- the values the runner reads -- and left alone otherwise; everything else is unchanged."""
    import fair_marl_b200 as fm
    cfg = FormationConfig(num_agents=3, num_obstacles=3, episode_length=6)
    e_all = fm.B200FormationVecEnv(_sim(cfg), num_envs=64, seed=3)
    e_end = fm.B200FormationVecEnv(_sim(cfg, info_every_step=False), num_envs=64, seed=3)
    e_all.reset_tensor(); e_end.reset_tensor()
    rng = np.random.default_rng(0)
    for t in range(13):
        a = _actions(rng.integers(0, 5, (64, 3)))
        o_all, o_end = _np(e_all.step_tensor(a)), _np(e_end.step_tensor(a))
        for k in ("obs", "node_obs", "adj_env", "reward", "done"):
            assert (o_all[k] == o_end[k]).all(), (t, k)
        fin = o_all["done"].all(axis=1)
        assert (o_all["info"][fin] == o_end["info"][fin]).all()
        if t < 5:
            assert (o_end["info"] == 0).all()                           # untouched before the first terminal step
    e_all.close(); e_end.close()


def test_partial_outputs_do_not_leave_ready_flags_behind():
    """A step without node_obs / adj runs the logic kernel alone (no image kernel to consume the per-16-env ready flags of the
    dependent launch); the steps after it must still build their rows from THEIR recipes."""
    import ctypes as C
    import torch
    import fair_marl_b200 as fm
    from fair_marl_b200 import _lib
    cfg = FormationConfig(num_agents=3, num_obstacles=3, episode_length=9)
    B = 4096
    e_a = fm.B200FormationVecEnv(_sim(cfg), num_envs=B, seed=5)
    e_b = fm.B200FormationVecEnv(_sim(cfg), num_envs=B, seed=5)
    e_a.reset_tensor(); e_b.reset_tensor()
    g = torch.Generator(device="cuda").manual_seed(1)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for t in range(12):
        a = torch.randint(0, 5, (B, 3), generator=g, device="cuda", dtype=torch.int32)
        o_b = e_b.step_tensor(a)
        if t % 3 == 1:                                  # logic kernel alone
            s = e_a._slots[0]
            o = _lib.FmOutputs(s["obs"].data_ptr(), None, None, s["reward"].data_ptr(), s["done"].data_ptr(), s["info"].data_ptr())
            _lib.check(e_a.lib.fm_formation_step(e_a._h, a.data_ptr(), C.byref(o), stream), "fm_formation_step")
            assert torch.equal(s["obs"], o_b["obs"]), t
        else:
            o_a = e_a.step_tensor(a)
            for k in ("obs", "node_obs", "adj_env", "reward"):
                assert torch.equal(o_a[k], o_b[k]), (t, k)
    e_a.close(); e_b.close()


# ---- launch variants -------------------------------------------------------------------------------------------------
# FM_FORM_PDL=0 (image kernel in plain stream order), FM_FORM_PREFETCH=0 (every reset drawn inline instead of copied from the
# pending block the side stream prefetched), FM_FORM_FUSED=1 (one generic kernel instead of logic + image): each must give
# the same bytes as the default.  With the prefetch on, an env that resets again within two steps takes the inline draw
# or the pending block depending on how the side stream's kernel interleaves with the step: the two must not differ either.
FORM_SWITCHES = ("FM_FORM_PDL", "FM_FORM_PREFETCH", "FM_FORM_FUSED", "FM_FORM_LANES")
LAUNCH_VARIANTS = {"pdl_off": {"FM_FORM_PDL": "0"}, "prefetch_off": {"FM_FORM_PREFETCH": "0"},
                   "pdl_and_prefetch_off": {"FM_FORM_PDL": "0", "FM_FORM_PREFETCH": "0"}, "fused": {"FM_FORM_FUSED": "1"}}


def _scripted_session(N, O, monkeypatch):
    """Every output and the whole state after each call of: reset; goal-seeking single steps with episode_length 1, 2 and 3
    (every env resets on every step, every other step, ...); a masked reset in mid-episode; rollout_tensor with one lane and
    with two (B >= 4096); a rollout_tensor captured in a CUDA graph and replayed twice.  B = 4096 + 45: ragged tiles."""
    import torch
    import fair_marl_b200 as fm
    B, T = 4096 + 45, 4
    assignment = ("fair", "optimal", "random")[(N + O) % 3]
    rng = np.random.default_rng(3)
    g = torch.Generator(device="cuda").manual_seed(4)
    rec = []

    def snap(label, env, out):
        d = {k: v.clone() for k, v in out.items()}
        d.update({"state." + k: v for k, v in env.get_state().items()})
        rec.append((label, d))

    def slots(label, env, slot_of):
        for t, k in enumerate(slot_of):
            rec.append(((label, t), {name: v.clone() for name, v in env.slot_outputs(k).items()}))
        snap((label, "state"), env, {})

    for L in (1, 2, 3):
        cfg = FormationConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=L,
                              fairness_reward=assignment == "fair", assignment=assignment)
        env = fm.B200FormationVecEnv(_sim(cfg), num_envs=B, seed=L, env_offset=5)
        snap(("reset", L), env, env.reset_tensor())
        for t in range(6):
            snap(("step", L, t), env, env.step_tensor(_actions(_goal_seeking(_from_device(env.get_state()), rng))))
            if L == 3 and t == 1:                                       # step 2 of 3 of the first episode
                snap(("masked reset", L), env, env.reset_tensor(rng.random(B) < 0.3))
        env.close()
    cfg = FormationConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=2,
                          fairness_reward=assignment == "fair", assignment=assignment)
    env = fm.B200FormationVecEnv(_sim(cfg, info_every_step=False), num_envs=B, seed=9, num_slots=T)
    env.reset_tensor()
    slots("rollout", env, env.rollout_tensor(torch.randint(0, 5, (T, B, N), generator=g, device="cuda", dtype=torch.int32)))
    monkeypatch.setenv("FM_FORM_LANES", "2")
    slots("two lanes", env, env.rollout_tensor(torch.randint(0, 5, (T, B, N), generator=g, device="cuda", dtype=torch.int32)))
    monkeypatch.delenv("FM_FORM_LANES")
    acts = torch.randint(0, 5, (T, B, N), generator=g, device="cuda", dtype=torch.int32)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        slot_of = env.rollout_tensor(acts)
    for replay in range(2):
        graph.replay()
        slots(("graph replay", replay), env, slot_of)
    torch.cuda.synchronize()
    env.close()
    return rec


@pytest.mark.parametrize("N,O", SPLIT_GRID)
def test_launch_variants_are_bitwise_identical(N, O, monkeypatch):
    import torch
    for k in FORM_SWITCHES:
        monkeypatch.delenv(k, raising=False)
    ref = _scripted_session(N, O, monkeypatch)
    for name, switches in LAUNCH_VARIANTS.items():
        for k in FORM_SWITCHES:
            monkeypatch.delenv(k, raising=False)
        for k, v in switches.items():
            monkeypatch.setenv(k, v)
        got = _scripted_session(N, O, monkeypatch)
        assert [label for label, _ in got] == [label for label, _ in ref]
        for (label, a), (_, b) in zip(ref, got):
            for k in a:
                assert torch.equal(a[k], b[k]), (name, label, k)
        del got


# ---- masked reset ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,O,W,B", [(3, 2, 0, 45), (6, 4, 0, 37), (3, 3, 1, 33)])   # split / fused steps before, walls
def test_masked_reset_matches_oracle(N, O, W, B):
    """reset(mask) in mid-episode against FormationOracle.reset(mask): the envs with mask 1 draw a new episode (bit for bit:
    positions, goals, obstacles, walls, assignment); the others are re-observed, which rewrites their goal-occupancy table
    and goal history.  Outputs and the whole post-state of every env within tolerance, discrete state exact."""
    import fair_marl_b200 as fm
    cfg = FormationConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=20, num_walls=W,
                          fairness_reward=True)
    env = fm.B200FormationVecEnv(_sim(cfg), num_envs=B, seed=21, env_offset=2)
    orc = FormationOracle(cfg, B, seed=21, env_offset=2)
    env.reset_tensor()
    rng = np.random.default_rng(8)
    for t in range(5):
        env.step_tensor(_actions(_goal_seeking(_from_device(env.get_state()), rng)))
    dev = env.get_state()
    pre = _from_device(dev)
    assert pre.status.any()                                          # latches to clear or keep
    orc.set_state(pre)
    _walls_from_device(orc, dev)
    mask = rng.random(B) < 0.4
    mask[:2] = (True, False)
    out, ref = _np(env.reset_tensor(mask.astype(np.uint8))), orc.reset(mask)
    dev = env.get_state()
    post, rpost = _from_device(dev), orc.get_state()
    for f in ("pos", "landmark_pos", "obstacle_pos", "goal_match"):
        assert (getattr(post, f)[mask] == getattr(rpost, f)[mask]).all(), f
        assert (getattr(post, f)[~mask] == getattr(pre, f)[~mask]).all(), f
    if W:
        assert (dev["wall_axis"].cpu().numpy() == orc.wall_axis.astype(np.float32)).all()
        assert (dev["wall_orient"].cpu().numpy() == orc.wall_orient).all()
        assert (dev["wall_len"].cpu().numpy() == orc.wall_len.astype(np.float32)).all()
    for f in ("goal_match", "step", "episode", "status"):
        assert (getattr(post, f) == getattr(rpost, f)).all(), f
    assert (post.episode == pre.episode + mask).all()
    assert_close(out["obs"], ref["obs"], "obs")
    assert_close(out["node_obs"], ref["node_obs"], "node_obs")
    assert_close(out["adj_env"], ref["adj"], "adj")
    for f in fields(FormationState):
        if f.name not in INT_FIELDS and f.name != "status":
            assert_close(getattr(post, f.name), getattr(rpost, f.name), f.name)
    env.close()


# ---- alignment and partial outputs -----------------------------------------------------------------------------------
@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("B", [64, 45])
def test_outputs_at_any_alignment_and_partial_outputs(B, fused, monkeypatch):
    """The formation kernels write full, 16-byte aligned tiles through TMA bulk stores and everything else by lanes.  Output
    arrays 4, 8 or 12 bytes past a 16-byte boundary, and FmOutputs with null members (the ABI allows any subset; without
    node_obs and adj the split path runs the logic kernel alone), must give the same bytes as the aligned full run, for
    reset, step and step_many."""
    import ctypes as C
    import torch
    import fair_marl_b200 as fm
    from fair_marl_b200 import _lib
    if fused:
        monkeypatch.setenv("FM_FORM_FUSED", "1")
    N, O = 3, 2
    E = 2 * N + O
    cfg = FormationConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=3)
    shapes = {"obs": (B, N, 11), "node_obs": (B, N, E, 13), "adj": (B, E, E), "reward": (B, N), "info": (B, N, 14)}
    everything = tuple(shapes) + ("done",)
    g = torch.Generator(device="cuda").manual_seed(6)
    acts = torch.randint(0, 5, (6, B, N), generator=g, device="cuda", dtype=torch.int32)

    def buffers(offset):
        out = {}
        for name, shp in shapes.items():
            n = int(np.prod(shp))
            out[name] = torch.full((n + 4,), float("nan"), device="cuda")[offset:offset + n].view(shp)
        out["done"] = torch.full((B * N + 4,), 7, dtype=torch.uint8, device="cuda")[offset:offset + B * N].view(B, N)
        return out

    def fm_outputs(out, keep):
        o = _lib.FmOutputs()
        for name in keep:
            setattr(o, name, out[name].data_ptr())
        return o

    def run(offset, keep):
        env = fm.B200FormationVecEnv(_sim(cfg), num_envs=B, seed=13)
        stream, rec = env._stream(), []
        out = buffers(offset)
        _lib.check(env.lib.fm_formation_reset(env._h, None, C.byref(fm_outputs(out, keep)), stream), "fm_formation_reset")
        rec.append({k: out[k].clone() for k in keep if k in ("obs", "node_obs", "adj")})
        for t in range(3):
            out = buffers(offset)
            _lib.check(env.lib.fm_formation_step(env._h, acts[t].data_ptr(), C.byref(fm_outputs(out, keep)), stream), "fm_formation_step")
            rec.append({k: out[k].clone() for k in keep})
        outs = [buffers(offset) for _ in range(3)]
        many = (_lib.FmOutputs * 3)(*[fm_outputs(o, keep) for o in outs])
        _lib.check(env.lib.fm_formation_step_many(env._h, acts[3].data_ptr(), 3, many, stream), "fm_formation_step_many")
        rec += [{k: o[k].clone() for k in keep} for o in outs]
        rec.append({k: v.clone() for k, v in env.get_state().items()})
        env.close()
        return rec

    ref = run(0, everything)
    assert all(not v.isnan().any() for r in ref[1:-1] for k, v in r.items() if v.is_floating_point())
    for offset, keep in [(1, everything), (2, everything), (3, everything), (0, ("adj",)), (3, ("adj",)), (0, ("node_obs",)),
                         (1, ("node_obs",)), (0, ("obs", "reward")), (2, ("obs", "reward")), (0, ("done", "info")), (3, ("done", "info"))]:
        got = run(offset, keep)
        for t, (a, b) in enumerate(zip(ref, got)):
            for k in b:
                assert torch.equal(a[k], b[k]), (offset, keep, t, k)


# ---- rejection-sampling cap ------------------------------------------------------------------------------------------
def test_reset_at_the_rejection_cap_matches_oracle():
    """world_size 0.05: every candidate position is within 2 (r + r) of an obstacle, so no placement is ever accepted and
    every agent of every env is placed by the MAX_DRAWS cap (4096 draws) -- bit for bit like the oracle -- followed by two
    steps (whose auto-resets hit the cap again) within tolerance."""
    import fair_marl_b200 as fm
    N, O, B = 2, 1, 3
    cfg = FormationConfig(num_agents=N, num_obstacles=O, world_size=0.05, goal_rew=30.0, collision_rew=30.0)
    env = fm.B200FormationVecEnv(_sim(cfg), num_envs=B, seed=3, env_offset=11)
    orc = FormationOracle(cfg, B, seed=3, env_offset=11)
    out, ref = _np(env.reset_tensor()), orc.reset()
    st, rs = _from_device(env.get_state()), orc.get_state()
    for f in ("pos", "landmark_pos", "obstacle_pos", "goal_match"):
        assert (getattr(st, f) == getattr(rs, f)).all(), f
    assert all(orc._obstacle_collision(b, st.pos[b, i]) for b in range(B) for i in range(N))   # accepted by the cap alone
    assert_close(st.min_time, rs.min_time, "min_time")
    assert_close(out["obs"], ref["obs"], "reset obs")
    assert_close(out["node_obs"], ref["node_obs"], "reset node_obs")
    assert_close(out["adj_env"], ref["adj"], "reset adj")
    rng = np.random.default_rng(2)
    for t in range(2):
        cur = _from_device(env.get_state())
        orc.set_state(cur)
        a = _goal_seeking(cur, rng)
        out = _np(env.step_tensor(_actions(a)))
        ref = orc.step(a, autoreset=True)
        post, rpost = _from_device(env.get_state()), orc.get_state()
        _compare_step(out, ref, post, rpost)
        hit = ref["reset"]
        assert (post.pos[hit] == rpost.pos[hit]).all() and (post.landmark_pos[hit] == rpost.landmark_pos[hit]).all()
        assert_close(post.pos, rpost.pos, "pos")
    env.close()
