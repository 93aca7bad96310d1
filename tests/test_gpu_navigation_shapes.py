"""Navigation kernels at the shapes the hand-picked parity cases of test_gpu_parity.py never reach.

* Every group size G of the group-per-env kernels (step / reset / prefetch_kernel<G, WALLS>, fm_kernels.cu) with and
  without walls, up to the largest entity table fm_create accepts for that G (shared memory), with a case that runs the
  runtime tail loop of distance_tile (fm_device.cuh: more landmark / obstacle pairs than SD_MAX x G).
* Every agent-warp shape (FM_AW_CASES, fm_aw.cuh) with relative and with global node features, stepped against the
  oracle, and its launch variants (FM_ROLL=1: aw_roll_kernel, FM_PREFETCH=2) compared bit for bit.
* The config constants (world_size, max_speed, min_dist_thresh, fair_rew / zeroshift, goal_rew / collision_rew), the
  MAX_DRAWS cap of the rejection sampling, and the edge list at E = 39 ... 115.

tests/conftest.py runs every case under both kernel mappings.  A shape without agent-warp kernels runs the group-per-env
kernels under either, so its 'auto' run is skipped as a duplicate of its 'group' run.
"""
import os
import re

import numpy as np
import pytest

from oracle.edges import process_adj as oracle_process_adj
from oracle.navgraph import INFO_KEYS, NavConfig, NavGraphOracle
from parity_util import assert_close, assert_fairness_close, compare_step_outputs, device_state_to_nav, sim_config_from

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "fair-marl_b200", "csrc")


# ------------------------------------------------------------------------------------------------ compiled shapes
def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _aw_cases():
    """(N, O) of FM_AW_CASES and (N, O, W) of FM_AW_WALL_CASES, parsed from fm_aw.cuh."""
    src = _read("fm_aw.cuh")
    plain = re.search(r"#define FM_AW_CASES\(X\)(.*)", src).group(1)
    walls = re.search(r"#define FM_AW_WALL_CASES\(X\)(.*)", src).group(1)
    return ([tuple(map(int, m)) for m in re.findall(r"X\((\d+), (\d+)\)", plain)],
            [tuple(map(int, m)) for m in re.findall(r"X\((\d+), (\d+), (\d+)\)", walls)])


def _sd_max(G, walls):
    """SD_MAX of distance_tile<G, WALLS> (fm_device.cuh): the landmark / obstacle pairs per lane kept in registers.
    The right-hand side is a nest of `cond ? a : b` over `G == n` and `WALLS`, evaluated here."""
    expr = re.search(r"constexpr int SD_MAX = ([^;]+);", _read("fm_device.cuh")).group(1)
    toks = re.findall(r"\d+|==|[?:()]|\w+", expr)
    pos = 0

    def take():
        nonlocal pos
        pos += 1
        return toks[pos - 1]

    def atom():
        t = take()
        if t == "(":
            v = ternary()
            assert take() == ")"
            return v
        if t == "WALLS":
            return int(walls)
        if t == "G":
            assert take() == "=="
            return int(G == int(take()))
        return int(t)

    def ternary():
        c = atom()
        if pos < len(toks) and toks[pos] == "?":
            take()
            a = ternary()
            assert take() == ":"
            b = ternary()
            return a if c else b
        return c

    v = ternary()
    assert pos == len(toks), expr
    return v


def group_size(n):
    """fm_kernels.cu group_size: lanes per env of the group-per-env kernels."""
    return 4 if n <= 4 else (8 if n <= 8 else (16 if n <= 16 else 32))


def static_pairs(N, O, W):
    M = N + O + W
    return M * (M - 1) // 2


def group_smem_bytes(N, O, W):
    """Dynamic shared memory of one CTA (4 warps) of the group-per-env kernels, as fm_create sizes it (fm_abi.cu)."""
    r4 = lambda x: (x + 3) & ~3
    E, EPW = 2 * N + O + W, 32 // group_size(N)
    per_warp = (r4(EPW * E * 8) + r4(max(EPW * E * E + 3, 2 * (32 * 11 + 4))) + r4(EPW * N * 7 + 3) + r4(EPW * N))
    return per_warp * 4 * 4


SMEM_LIMIT = 227 * 1024


def largest_obstacles(N, W):
    return max(O for O in range(65) if group_smem_bytes(N, O, W) <= SMEM_LIMIT)


AW_CASES, AW_WALL_CASES = _aw_cases()


def _is_aw(N, O, W, feat="relative"):
    return (N, O) in AW_CASES if W == 0 else (N, O, W) in AW_WALL_CASES and feat == "relative"


def _skip_auto_duplicate(N, O, W, feat="relative"):
    import parity_util
    if parity_util.MAPPING == "auto" and not _is_aw(N, O, W, feat):
        pytest.skip("no agent-warp kernels at this shape: 'auto' runs the same group-per-env kernels as 'group'")


def _run_once():
    import parity_util
    if parity_util.MAPPING == "auto":
        pytest.skip("does not depend on the kernel mapping: runs under 'group' only")


# ------------------------------------------------------------------------------------------------ device helpers
def _env(cfg, B, seed=7, env_offset=3, **sim):
    import fair_marl_b200 as fm
    return fm.B200GraphVecEnv(sim_config_from(cfg, **sim), num_envs=B, seed=seed, env_offset=env_offset)


def _np(out):
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in out.items()}


def _actions(a):
    import torch
    return torch.as_tensor(np.asarray(a), dtype=torch.int32, device="cuda")


def _mask(m):
    import torch
    return torch.as_tensor(np.asarray(m, dtype=np.uint8), device="cuda")


def _seek_actions(st, rng, p_random=0.25):
    """oracle/make_golden.py::_seek_actions over the batch: greedy move towards the assigned goal, a uniform action
    with probability p_random."""
    goal = np.take_along_axis(st.landmark_pos, st.goal_match[..., None], axis=1)
    d = goal - st.pos
    a = np.where(np.abs(d[..., 0]) > np.abs(d[..., 1]), np.where(d[..., 0] > 0, 1, 2), np.where(d[..., 1] > 0, 3, 4))
    return np.where(rng.random(a.shape) < p_random, rng.integers(0, 5, a.shape), a)


def _assert_placements_equal(post, rpost, sel, W):
    for f in ("pos", "landmark_pos", "obstacle_pos", "goal_match"):
        assert (getattr(post, f)[sel] == getattr(rpost, f)[sel]).all(), f
    if W:
        assert (post.wall_axis[sel] == rpost.wall_axis[sel].astype(np.float32)).all()
        assert (post.wall_orient[sel] == rpost.wall_orient[sel]).all()
        assert (post.wall_len[sel] == rpost.wall_len[sel].astype(np.float32)).all()


def _compare_info(info_dev, info_ref):
    for k, key in enumerate(INFO_KEYS):
        if key in ("Mean_by_variance", "Time_mean_by_stddev"):
            assert_fairness_close(info_dev[..., k], info_ref[key], key)
        else:
            assert_close(info_dev[..., k], info_ref[key], key)


def _rollout_matches_oracle(cfg: NavConfig, B: int, episodes: int = 2, seed: int = 7, env_offset: int = 3):
    """Reset, a masked reset and `episodes` episodes of goal-seeking steps (25 % random actions), the oracle re-synced to
    the device state before every step.  Returns what happened (per-event counts and the oracle's reward / speed
    extremes) so that each case can assert that the events it exists for took place."""
    N, O, W = cfg.num_agents, cfg.num_obstacles, cfg.num_walls
    env = _env(cfg, B, seed, env_offset, info_every_step=True)
    assert env.num_entities == cfg.num_entities
    orc = NavGraphOracle(cfg, B, seed=seed, env_offset=env_offset)
    if cfg.max_speed is None:                    # no side writes min_time then: start from the device's zeroed block
        orc.s.min_time[:] = device_state_to_nav(env.get_state()).min_time
    out, ref = _np(env.reset_tensor()), orc.reset()
    st, rs = device_state_to_nav(env.get_state()), orc.get_state()
    _assert_placements_equal(st, rs, slice(None), W)
    assert (st.episode == 1).all() and (st.step == 0).all() and (st.vel == 0).all()
    assert_close(st.min_time, rs.min_time, "reset min_time")
    assert_close(out["obs"][..., :6], ref["obs"][..., :6], "reset obs")
    assert_fairness_close(out["obs"][..., 6], ref["obs"][..., 6])
    assert_close(out["node_obs"], ref["node_obs"], "reset node_obs")
    assert_close(out["adj_env"], ref["adj"], "reset adj")
    rng = np.random.default_rng(5)
    ev = dict(agent_coll=0, obst_coll=0, latch=0, resets=0, clip_lo=0, above_coll_clip=0, fair_wide=0, max_speed=0.0,
              reset_extent=float(np.abs(st.pos).max()))
    rew_sum, info_sum = np.zeros(N), np.zeros((N, 14))
    steps = episodes * cfg.episode_length
    masked_at = cfg.episode_length // 2
    for t in range(steps):
        if t == masked_at:                       # a masked reset in the middle of an episode: envs 1, 4, 7, ... restart
            mask = np.arange(B) % 3 == 1
            orc.set_state(device_state_to_nav(env.get_state()))
            out = _np(env.reset_tensor(mask=_mask(mask)))
            ref = orc.reset(mask=mask)
            _assert_placements_equal(device_state_to_nav(env.get_state()), orc.get_state(), mask, W)
            assert_close(out["obs"][..., :6], ref["obs"][..., :6], "masked reset obs")
            assert_close(out["node_obs"], ref["node_obs"], "masked reset node_obs")
            assert_close(out["adj_env"], ref["adj"], "masked reset adj")
        cur = device_state_to_nav(env.get_state())
        orc.set_state(cur)
        a = _seek_actions(cur, rng)
        out = _np(env.step_tensor(_actions(a)))
        ref = orc.step(actions=a, autoreset=True)
        out["adj"] = out["adj_env"]
        compare_step_outputs(out, ref, cfg)
        _compare_info(out["info"], ref["info"])
        post, rpost = device_state_to_nav(env.get_state()), orc.get_state()
        hit = ref["reset"]
        assert (out["done"].astype(bool) == hit[:, None]).all()
        if hit.any():
            _assert_placements_equal(post, rpost, hit, W)
            assert (post.step[hit] == 0).all() and (post.episode == rpost.episode).all()
        assert_close(post.pos, rpost.pos, "pos")
        assert_close(post.vel, rpost.vel, "vel")
        assert_close(post.min_time, rpost.min_time, "min_time")
        for f in ("num_agent_collisions", "num_obstacle_collisions", "step"):
            assert (getattr(post, f) == getattr(rpost, f)).all(), f
        info = ref["info"]
        ev["agent_coll"] += int((info["Num_agent_collisions"] > 0).sum())
        ev["obst_coll"] += int((info["Num_obst_collisions"] > 0).sum())
        ev["latch"] += int((info["Time_req_to_goal"] != -1).sum())
        ev["resets"] += int(hit.sum())
        ev["clip_lo"] += int((ref["reward"] == -2 * cfg.collision_rew).sum())
        ev["above_coll_clip"] += int((ref["reward"] > cfg.collision_rew + cfg.fair_rew).sum())
        if cfg.fairness_reward:                  # obs[6] is the reward's fairness_param (but not on a reset's rows)
            fair = cfg.fair_rew * np.tanh(ref["obs"][~hit, :, 6] - cfg.zeroshift)
            ev["fair_wide"] += int((np.abs(fair) > 1).sum())
        ev["max_speed"] = max(ev["max_speed"], float(np.sqrt((cur.vel ** 2).sum(-1)).max()))
        rew_sum += ref["reward"].sum(0)
        for k, key in enumerate(INFO_KEYS):
            info_sum[:, k] += info[key][hit].sum(0)
    v = env.read_stats().cpu().numpy()
    np.testing.assert_allclose(v[:N], rew_sum, rtol=1e-5, atol=1e-3)
    got = v[N:15 * N].reshape(N, 14)
    for k, key in enumerate(INFO_KEYS):
        if "by" not in key:                      # the two ill-conditioned ratios are compared per step above
            np.testing.assert_allclose(got[:, k], info_sum[:, k], rtol=2e-5, atol=1e-3, err_msg=key)
    assert v[15 * N] == ev["resets"] and v[15 * N + 1] == steps * B
    env.close()
    assert ev["resets"] >= B
    return ev


def _assert_events(ev, cfg, latch=True):
    if cfg.num_agents > 1:
        assert ev["agent_coll"] > 0, ev
    if cfg.num_obstacles > 0 or cfg.num_walls > 0:
        assert ev["obst_coll"] > 0, ev
    if latch:
        assert ev["latch"] > 0, ev


# ------------------------------------------------------------------------------------------------ 1. group-per-env shapes
# (N, O, W, B, options).  B is ragged for the group's envs per warp (32 / G); G = 32 holds one env per warp.
GROUP_CASES = [
    (3, 8, 0, 45, {}),                           # G = 4: tail loop (55 pairs > 12 x 4)
    (4, 30, 0, 9, {}),                           # G = 4: largest E without walls
    (4, 28, 2, 17, {}),                          # G = 4: largest E with walls
    (8, 0, 0, 37, {}),                           # G = 8: full group
    (8, 3, 0, 29, {}),                           # G = 8: tail loop (55 pairs > 6 x 8)
    (7, 4, 0, 22, {}),                           # G = 8: tail loop
    (8, 39, 0, 7, {}),                           # G = 8: largest E
    (8, 37, 2, 6, {}),                           # G = 8 with walls: largest E, tail loop (1081 pairs > 9 x 8)
    (6, 5, 0, 13, {"graph_feat_type": "global"}),
    (9, 0, 0, 21, {}),                           # G = 16: 7 idle lanes
    (16, 5, 0, 11, {}),                          # G = 16: tail loop (210 pairs > 12 x 16)
    (16, 48, 0, 3, {}),                          # G = 16: largest E
    (16, 46, 2, 4, {}),                          # G = 16 with walls: largest E
    (12, 3, 0, 5, {"graph_feat_type": "global"}),
    (10, 2, 0, 9, {"collaborative": True}),
    (17, 0, 0, 13, {}),                          # G = 32
    (32, 0, 0, 5, {}),                           # G = 32: full warp, tail loop (496 pairs > 12 x 32)
    (17, 64, 0, 3, {}),                          # G = 32: O at the ABI limit
    (32, 51, 0, 2, {}),                          # G = 32: largest E (115)
    (24, 3, 2, 4, {}),                           # G = 32 with walls, tail loop (406 pairs)
    (20, 4, 0, 5, {"graph_feat_type": "global"}),
    (18, 1, 0, 6, {"collaborative": True}),
    (21, 2, 0, 1, {"fairness_reward": False}),   # B = 1
]


def _case_id(c):
    N, O, W, B, opt = c
    return f"{N}-{O}-{W}-{B}" + "".join(f"-{v if isinstance(v, str) else k}" for k, v in opt.items())


@pytest.mark.gpu
@pytest.mark.parametrize("case", GROUP_CASES, ids=_case_id)
def test_group_shapes_match_oracle(case):
    N, O, W, B, opt = case
    _skip_auto_duplicate(N, O, W, opt.get("graph_feat_type", "relative"))
    cfg = NavConfig(num_agents=N, num_obstacles=O, num_walls=W, episode_length=8, **opt)
    _assert_events(_rollout_matches_oracle(cfg, B), cfg)


@pytest.mark.gpu
@pytest.mark.parametrize("feat", ["relative", "global"])
@pytest.mark.parametrize("N,O,B", [(1, 1, 70), (2, 0, 45), (3, 0, 33), (3, 3, 100), (4, 2, 37)])
def test_agent_warp_shapes_match_oracle(N, O, B, feat):
    """Every FM_AW_CASES shape under both node feature types, against the oracle itself.  'auto' runs aw_kernel<N, O, ·, NF>,
    'group' the group-per-env kernels at G = 4."""
    import parity_util
    cfg = NavConfig(num_agents=N, num_obstacles=O, episode_length=8, graph_feat_type=feat)
    ev = _rollout_matches_oracle(cfg, B, episodes=3)
    _assert_events(ev, cfg)
    env = _env(cfg, 1)
    assert env.mapping == ("aw" if parity_util.MAPPING == "auto" else "group")
    env.close()


# ------------------------------------------------------------------------------------------------ 2. shape limits
@pytest.mark.gpu
@pytest.mark.parametrize("N,O,W", [(4, 31, 0), (8, 40, 0), (16, 49, 0), (32, 52, 0), (4, 29, 2), (8, 38, 2)])
def test_shapes_past_the_shared_memory_limit_are_refused(N, O, W):
    """One obstacle past the largest entity table of each group size needs more than 227 KB of shared memory per CTA:
    fm_create refuses it, and accepts the shape with one obstacle less."""
    import fair_marl_b200 as fm
    assert O == largest_obstacles(N, W) + 1
    _skip_auto_duplicate(N, O, W)
    with pytest.raises(fm._lib.FairMarlError, match="shared memory"):
        _env(NavConfig(num_agents=N, num_obstacles=O, num_walls=W), 3)
    env = _env(NavConfig(num_agents=N, num_obstacles=O - 1, num_walls=W), 3)
    env.reset_tensor()
    env.close()


@pytest.mark.gpu
def test_more_than_32_agents_or_64_obstacles_are_refused():
    import fair_marl_b200 as fm
    _run_once()
    with pytest.raises(fm._lib.FairMarlError, match="num_agents"):
        _env(NavConfig(num_agents=33, num_obstacles=0), 1)
    with pytest.raises(fm._lib.FairMarlError, match="num_obstacles"):
        _env(NavConfig(num_agents=17, num_obstacles=65), 1)


# ------------------------------------------------------------------------------------------------ 3. launch variants
@pytest.mark.gpu
@pytest.mark.parametrize("feat", ["relative", "global"])
@pytest.mark.parametrize("N,O", [(1, 1), (2, 0), (3, 0), (3, 3), (4, 2)])
def test_launch_variants_are_bitwise_identical(N, O, feat, monkeypatch):
    """A scripted session (single steps across auto-resets, a masked reset, rollout_tensor over an episode boundary, a
    second rollout) gives the same bytes under every launch variant of the mapping: agent-warp one-shot kernels
    (default), the persistent aw_roll_kernel (FM_ROLL=1) and the prefetched next episode (FM_PREFETCH=2); group-per-env
    with the prefetch (default) and with inline resets (FM_PREFETCH=0)."""
    import torch
    import parity_util
    variants = ({}, {"FM_ROLL": "1"}, {"FM_PREFETCH": "2"}) if parity_util.MAPPING == "auto" else ({}, {"FM_PREFETCH": "0"})
    cfg = NavConfig(num_agents=N, num_obstacles=O, episode_length=3, graph_feat_type=feat)
    B = 75
    runs = []
    for var in variants:
        for k in ("FM_ROLL", "FM_PREFETCH"):
            monkeypatch.delenv(k, raising=False)
        for k, v in var.items():
            monkeypatch.setenv(k, v)
        import fair_marl_b200 as fm
        env = fm.B200GraphVecEnv(sim_config_from(cfg, info_every_step=True), num_envs=B, seed=13, env_offset=2, num_slots=8)
        g = torch.Generator(device="cuda").manual_seed(8)
        rec = []

        def keep(o):
            rec.extend(o[k].clone() for k in ("obs", "node_obs", "adj_env", "reward", "done", "info") if k in o)

        keep(env.reset_tensor())
        for t in range(7):
            keep(env.step_tensor(torch.randint(0, 5, (B, N), generator=g, device="cuda", dtype=torch.int32)))
        keep(env.reset_tensor(mask=(torch.arange(B, device="cuda") % 4 == 1).to(torch.uint8)))
        for t in range(2):
            keep(env.step_tensor(torch.randint(0, 5, (B, N), generator=g, device="cuda", dtype=torch.int32)))
        for T in (7, 4):
            acts = torch.randint(0, 5, (T, B, N), generator=g, device="cuda", dtype=torch.int32)
            slots = env.rollout_tensor(acts)
            for i, slot in enumerate(slots):
                if slot not in slots[i + 1:]:
                    keep(env.slot_outputs(slot))
        st = env.get_state()
        rec.extend(st[k].clone() for k in sorted(st))
        rec.append(env.read_stats())
        runs.append(rec)
        env.close()
    for var, run in zip(variants[1:], runs[1:]):
        assert len(run) == len(runs[0])
        for k, (x, y) in enumerate(zip(runs[0], run)):
            assert torch.equal(x, y), (var, k)


# ------------------------------------------------------------------------------------------------ 4. parameter sweep
SWEEP = {
    "world_1.2": dict(world_size=1.2),
    "world_3.0": dict(world_size=3.0),
    "vmax_none": dict(max_speed=None),
    "vmax_0.7": dict(max_speed=0.7),
    "thresh_0.3": dict(min_dist_thresh=0.3),
    "fair_2.5_zs_2": dict(fair_rew=2.5, zeroshift=2.0),
    "goal_10_coll_3": dict(goal_rew=10.0, collision_rew=3.0),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SWEEP))
@pytest.mark.parametrize("N,O,B", [(3, 3, 200), (7, 3, 45), (20, 2, 11)])
def test_config_constants_match_oracle(N, O, B, name):
    """One config group away from its default at a time, on an agent-warp shape, at G = 8 and at G = 32; each asserts
    that the value it changes mattered in the run."""
    _skip_auto_duplicate(N, O, 0)
    opt = SWEEP[name]
    cfg = NavConfig(num_agents=N, num_obstacles=O, episode_length=8, **opt)
    ev = _rollout_matches_oracle(cfg, B, episodes=3)
    _assert_events(ev, cfg, latch=name != "world_3.0")
    if name == "vmax_none":
        assert ev["max_speed"] > 2.0, ev          # faster than the default clip would allow
    elif name == "vmax_0.7":
        assert 0.69 < ev["max_speed"] <= 0.7 * (1 + 1e-6), ev
    elif name == "world_3.0":
        assert ev["reset_extent"] > 1.0, ev      # placed outside the default world
    elif name == "world_1.2":
        assert ev["reset_extent"] <= 0.6, ev
    elif name == "thresh_0.3":
        assert ev["latch"] >= 3 * B, ev
    elif name == "fair_2.5_zs_2":
        assert ev["fair_wide"] > 0, ev           # fairness terms outside the [-1, 1] of fair_rew = 1
    elif name == "goal_10_coll_3":
        assert ev["clip_lo"] > 0, ev             # the lower clip bound -2 * collision_rew ...
        assert ev["above_coll_clip"] > 0, ev     # ... and rewards above collision_rew + fair_rew (the upper one is goal_rew + fair_rew)


# ------------------------------------------------------------------------------------------------ 5. rejection cap
@pytest.mark.gpu
@pytest.mark.parametrize("N,O,W,B", [(3, 3, 0, 40), (3, 3, 2, 33), (6, 2, 0, 13), (17, 2, 0, 3)])
def test_reset_at_the_rejection_cap_matches_oracle(N, O, W, B):
    """world_size = 0.05: every candidate overlaps an obstacle or an earlier slot, so each reset draws until the
    MAX_DRAWS cap accepts whatever it has.  The placements are bit-exact after the reset and after two steps with
    episode_length 1 (every step auto-resets: the group mapping takes the prefetched block)."""
    _skip_auto_duplicate(N, O, W)
    cfg = NavConfig(num_agents=N, num_obstacles=O, num_walls=W, world_size=0.05, episode_length=1)
    env = _env(cfg, B, seed=3, env_offset=9, info_every_step=True)
    orc = NavGraphOracle(cfg, B, seed=3, env_offset=9)
    out, ref = _np(env.reset_tensor()), orc.reset()
    _assert_placements_equal(device_state_to_nav(env.get_state()), orc.get_state(), slice(None), W)
    assert_close(out["node_obs"], ref["node_obs"], "reset node_obs")
    assert_close(out["adj_env"], ref["adj"], "reset adj")
    rng = np.random.default_rng(1)
    for t in range(2):
        cur = device_state_to_nav(env.get_state())
        orc.set_state(cur)
        a = rng.integers(0, 5, (B, N))
        out = _np(env.step_tensor(_actions(a)))
        ref = orc.step(actions=a, autoreset=True)
        assert ref["reset"].all()
        out["adj"] = out["adj_env"]
        compare_step_outputs(out, ref, cfg)
        _assert_placements_equal(device_state_to_nav(env.get_state()), orc.get_state(), slice(None), W)
    # the cap was what ended the rejection: placements closer than 1.05 * (r + r) were accepted
    st = orc.get_state()
    d = np.linalg.norm(st.pos[:, :, None] - st.pos[:, None, :], axis=-1) + np.eye(N) * 9
    assert (d < 0.105).any()
    env.close()


# ------------------------------------------------------------------------------------------------ 6. edge list
@pytest.mark.gpu
@pytest.mark.parametrize("form", ["stream", "three", "fused"])
@pytest.mark.parametrize("E", [39, 40, 100, 101, 108, 115])
def test_edge_list_at_large_entity_counts(E, form, monkeypatch):
    """fm_edge_list on full graphs (every entry is an edge: each entry index q < E^2 is split into row and column) and on
    random graphs, with repeat 1 and 3.  The fused form needs 96 KB of shared memory at E = 39 and falls back above; the
    streamed form divides by E with a 20-bit reciprocal, exact up to E = 100, and falls back to the three-kernel form
    above."""
    import torch
    import fair_marl_b200 as fm
    _run_once()
    monkeypatch.delenv("FM_EDGE_FUSED", raising=False)
    monkeypatch.setenv("FM_EDGE_FORM", form)
    rng = np.random.default_rng(E)
    full = (rng.random((5, E, E)) * 0.9 + 0.05).astype(np.float32)
    rand = (rng.random((37, E, E)) * 2).astype(np.float32)
    rand[3] = 0.0
    for adj, want_full in ((full, True), (rand, False)):
        for repeat in (1, 3):
            ei, ea = fm.process_adj(torch.as_tensor(adj, device="cuda"), 1.0, repeat=repeat)
            rei, rea = oracle_process_adj(np.repeat(adj, repeat, axis=0), 1.0)
            if want_full:
                assert rei.shape[1] == repeat * adj.shape[0] * E * E
            assert tuple(ei.shape) == rei.shape
            assert (ei.cpu().numpy() == rei).all() and (ea.cpu().numpy() == rea).all()


def test_edge_reciprocal_division_is_exact_up_to_e_100():
    """fm_edges.cu / fm_kernels.cu split an entry index q < E^2 into (q / E, q % E) as (q * ceil(2^20 / E)) >> 20 while
    E <= 100: exact for every such q.  At E = 108 it is not, which is why the larger tables take the division."""
    for E in range(1, 101):
        q = np.arange(E * E, dtype=np.uint64)
        magic = np.uint64(((1 << 20) + E - 1) // E)
        assert ((q * magic) >> np.uint64(20) == q // np.uint64(E)).all(), E
    q = np.arange(108 * 108, dtype=np.uint64)
    assert not ((q * np.uint64(((1 << 20) + 107) // 108)) >> np.uint64(20) == q // np.uint64(108)).all()


# ------------------------------------------------------------------------------------------------ 7. guard
def test_every_compiled_navigation_shape_has_a_case():
    """Fails when the case lists stop covering an agent-warp shape (with each node feature type, and in the launch-variant
    test), a group size with or without walls, a group size whose distance_tile tail loop (more static pairs than
    SD_MAX x G) no case enters, or the largest entity table of a group size."""
    assert AW_CASES and AW_WALL_CASES
    aw = {(n, o) for n, o, _ in _params_of(test_agent_warp_shapes_match_oracle, "N,O,B")}
    missing = [("agent-warp", c) for c in AW_CASES if c not in aw]
    missing += [("feature type", f) for f in ("relative", "global") if f not in _params_of(test_agent_warp_shapes_match_oracle, "feat")]
    variants = set(_params_of(test_launch_variants_are_bitwise_identical, "N,O"))
    missing += [("launch variants", c) for c in AW_CASES if c not in variants]
    group = [(N, O, W) for N, O, W, _, _ in GROUP_CASES]
    for G in (4, 8, 16, 32):
        mine = [s for s in group if group_size(s[0]) == G]
        for walls in (False, True):
            if not any((W > 0) == walls for _, _, W in mine):
                missing.append(("group size", G, "walls" if walls else "no walls"))
        if not any(static_pairs(*s) > _sd_max(G, s[2] > 0) * G for s in mine):
            missing.append(("tail loop", G))
        if not any(W == 0 and O == largest_obstacles(N, 0) for N, O, W in mine):
            missing.append(("largest entity table", G))
    assert not missing, missing


def _params_of(fn, argnames):
    for m in getattr(fn, "pytestmark", []):
        if m.name == "parametrize" and m.args[0] == argnames:
            return list(m.args[1])
    raise AssertionError(f"{fn.__name__} has no parametrize over {argnames}")
