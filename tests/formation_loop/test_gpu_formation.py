"""The formation family in the device rollout loop (RolloutCollector / DeviceRolloutBuffer over B200FormationVecEnv,
step_tensor(out=)) and its on-device episode statistics (fm_formation_stats_enable / fm_formation_stats_read), on the GPU.
Helpers and the oracle plumbing are those of tests/test_gpu_formation.py."""
import numpy as np
import pytest

from oracle.formation import FormationConfig, FormationOracle
from oracle.navgraph import INFO_KEYS
from parity_util import assert_close, assert_fairness_close
from test_gpu_formation import FORM_SWITCHES, RATIO_KEYS, _actions, _from_device, _goal_seeking, _sim

pytestmark = pytest.mark.gpu


# ---- device rollout loop: RolloutCollector / DeviceRolloutBuffer over B200FormationVecEnv ------------------------------
def _collector_parts(N, O, B, W=0, seed=5, **kw):
    """Env + random-init policy in the shape of the shipped formation actors (obs 11, node rows 13), logits scaled up so
    that the deterministic policy depends on the state."""
    import torch
    import fair_marl_b200 as fm
    cfg = fm.FormationSimConfig(num_agents=N, num_obstacles=O, num_walls=W, goal_rew=30.0, collision_rew=30.0, **kw)
    env = fm.B200FormationVecEnv(cfg, num_envs=B, seed=seed)
    pc = fm.PolicyConfig(num_agents=N, obs_dim=11, node_feat_dim=13)
    torch.manual_seed(0)
    actor, critic = fm.DenseGraphActor(pc).to(env.device).eval(), fm.DenseGraphCritic(pc).to(env.device).eval()
    with torch.no_grad():
        actor.action_out.weight.mul_(100.0)
    return fm, cfg, env, actor, critic


# (3, 3, 96): split path, B N a multiple of 16 (16-byte aligned slabs: bulk stores); (3, 3, 45): split, ragged last tile;
# (5, 2, 64): fused kernel (N > 4); (3, 2, 64) with 2 walls: fused kernel with wall rows
@pytest.mark.parametrize("N,O,B,W", [(3, 3, 96, 0), (3, 3, 45, 0), (5, 2, 64, 0), (3, 2, 64, 2)])
def test_collector_writes_buffer_in_place_and_replays_bitwise(N, O, B, W):
    """The formation step kernels write the DeviceRolloutBuffer slabs directly (step_tensor(out=...)); replaying the recorded
    actions through a second env reproduces every slab bit for bit, and the bookkeeping follows GMPERunner.insert with
    per-agent early dones: masks = 1 - done, RNN states zeroed at done, active_masks 1 where alive or the env is done."""
    import torch
    fm, cfg, env, actor, critic = _collector_parts(N, O, B, W)
    col = fm.RolloutCollector(env, actor, critic, deterministic=True)
    buf = col.buffer
    T, E = cfg.episode_length, cfg.num_entities
    col.warmup(); col.run()
    torch.cuda.synchronize()
    env2 = fm.B200FormationVecEnv(cfg, num_envs=B, seed=5)
    r = env2.reset_tensor()
    assert torch.equal(r["obs"], buf.obs[0]) and torch.equal(r["node_obs"], buf.node_obs[0]) and torch.equal(r["adj_env"], buf.adj_env[0])
    for t in range(T):
        o = env2.step_tensor(buf.actions_env[t])
        assert torch.equal(o["obs"], buf.obs[t + 1]), t
        assert torch.equal(o["node_obs"], buf.node_obs[t + 1]), t
        assert torch.equal(o["adj_env"], buf.adj_env[t + 1]), t
        assert torch.equal(o["reward"], buf.rewards[t, :, :, 0]), t
        assert torch.equal(o["done"], buf.dones[t].bool()), t
    done = buf.dones.bool().cpu()
    assert (done.any(-1) & ~done.all(-1)).any(), "no per-agent early done in the episode"
    assert done.all(-1).any()
    keep = (~done).float().unsqueeze(-1)
    assert torch.equal(buf.masks[1:].cpu(), keep)
    rnn = buf.rnn_states[1:].cpu()
    assert (rnn[done] == 0).all() and (rnn[~done] != 0).any()
    active = torch.where(done.all(-1, keepdim=True), torch.ones_like(keep[..., 0]), keep[..., 0]).unsqueeze(-1)
    assert torch.equal(buf.active_masks[1:].cpu(), active)
    assert (buf.active_masks[1:] == 0).any()
    assert torch.equal(buf.actions[:, :, :, 0], buf.actions_env.float())
    col.finish()
    assert torch.isfinite(buf.returns).all()
    env.close(); env2.close()


@pytest.mark.parametrize("N,O", [(3, 3), (5, 2)])            # split path (PDL + pending-reset prefetch on), fused kernel
def test_collector_captured_graph_equals_eager_episode(N, O):
    import torch
    runs = []
    for use_graph in (False, True):
        fm, cfg, env, actor, critic = _collector_parts(N, O, 128, seed=11, episode_length=10)
        col = fm.RolloutCollector(env, actor, critic, deterministic=True)
        col.warmup(); col.run(); col.buffer.after_update()
        if use_graph:
            col.capture()
        col.run(); col.buffer.after_update(); col.run()
        torch.cuda.synchronize()
        b = col.buffer
        runs.append([x.clone() for x in (b.obs, b.node_obs, b.adj_env, b.rewards, b.dones, b.actions_env, b.rnn_states, b.masks,
                                         b.active_masks, b.value_preds, b.action_log_probs)])
        assert b.dones.bool().all(-1).any()                      # resets inside the captured episodes
        env.close()
    for x, y in zip(*runs):
        assert torch.equal(x, y)


def test_collector_fused_policy_equals_dense_on_formation_outputs():
    """The fused graph network (E = 9, 13 features, obs 11) against the dense torch modules on formation outputs: same
    actions, hence the same trajectories; values within 2e-5."""
    import torch
    outs = []
    for fused in (True, False):
        fm, cfg, env, actor, critic = _collector_parts(3, 3, 160, seed=11, episode_length=8)
        col = fm.RolloutCollector(env, actor, critic, deterministic=True, fused=fused)
        assert col.fused is fused
        col.warmup(); col.run()
        torch.cuda.synchronize()
        outs.append((col.buffer.actions_env.clone(), col.buffer.value_preds.clone(), col.buffer.obs.clone()))
        env.close()
    assert torch.equal(outs[0][0], outs[1][0])
    assert torch.equal(outs[0][2], outs[1][2])
    v0, v1 = outs[0][1].double(), outs[1][1].double()
    err = ((v0 - v1).abs() / v1.abs().clamp(min=1.0)).max().item()
    assert err <= 2e-5, err


def test_step_tensor_out_validation_and_collector_dims():
    import torch
    import fair_marl_b200 as fm
    B, N, O = 32, 3, 3
    E = 2 * N + O
    env = fm.B200FormationVecEnv(fm.FormationSimConfig(num_agents=N, num_obstacles=O), num_envs=B, seed=1, num_slots=2)
    buf = fm.DeviceRolloutBuffer(25, B, N, E, obs_dim=11, node_feat_dim=13, device=env.device)
    r = env.reset_tensor(out=buf.env_views(0, with_step=False))
    assert r["obs"].data_ptr() == buf.obs[0].data_ptr() and set(r) == {"obs", "node_obs", "adj_env"}
    a = torch.zeros(B, N, dtype=torch.int32, device=env.device)
    slot = env._slot
    o = env.step_tensor(a, out=buf.env_views(1))
    assert env._slot == slot                                             # the ring does not advance
    assert set(o) == set(env.step_tensor(a)) and o["done"].dtype == torch.bool
    assert o["reward"].data_ptr() == buf.rewards[0].data_ptr() and o["adj_env"].data_ptr() == buf.adj_env[1].data_ptr()
    bad_cases = []
    v = buf.env_views(1); v["adj"] = buf.adj[1]; bad_cases.append(v)                                  # expanded [B,N,E,E]
    v = buf.env_views(1); v["obs"] = buf.obs[1][:, :2]; bad_cases.append(v)                            # shape
    v = buf.env_views(1); v["done"] = buf.dones[0].bool(); bad_cases.append(v)                         # dtype
    v = buf.env_views(1); v["reward"] = torch.zeros(N, B, device=env.device).t(); bad_cases.append(v)  # not contiguous
    v = buf.env_views(1); del v["node_obs"]; bad_cases.append(v)                                       # missing
    for v in bad_cases:
        with pytest.raises(ValueError):
            env.step_tensor(a, out=v)
    with pytest.raises(ValueError):
        env.reset_tensor(out={**buf.env_views(0, with_step=False), "node_obs": buf.node_obs[0].transpose(1, 2)})
    actor = fm.DenseGraphActor(fm.PolicyConfig(num_agents=N)).to(env.device)           # navigation shape: obs 7, rows 11
    critic = fm.DenseGraphCritic(fm.PolicyConfig(num_agents=N)).to(env.device)
    with pytest.raises(ValueError):
        fm.RolloutCollector(env, actor, critic)
    env.close()


# ---- episode statistics -----------------------------------------------------------------------------------------------
def _keep_outputs(out, keep):
    from fair_marl_b200 import _lib
    o = _lib.FmOutputs()
    for name in keep:
        setattr(o, name, out[name].data_ptr())
    return o


def _stats_run(cfg, B, actions, keep=("obs", "node_obs", "adj", "reward", "done", "info"), stats=True, seed=7, env_offset=0):
    """reset + one fm_formation_step per row of `actions` [T,B,N] with FmOutputs members `keep` only; returns the stats
    vector (None with stats off), the per-step outputs of the kept members (host) and the final state."""
    import ctypes as C
    import torch
    import fair_marl_b200 as fm
    from fair_marl_b200 import _lib
    env = fm.B200FormationVecEnv(cfg, num_envs=B, seed=seed, env_offset=env_offset, episode_stats=stats)
    N, E = cfg.num_agents, cfg.num_entities
    env.reset_tensor()
    shapes = {"obs": (B, N, 11), "node_obs": (B, N, E, 13), "adj": (B, E, E), "reward": (B, N), "info": (B, N, 14)}
    out = {k: torch.zeros(s, device="cuda") for k, s in shapes.items()}
    out["done"] = torch.zeros((B, N), dtype=torch.uint8, device="cuda")
    stream, rec = env._stream(), []
    for t in range(actions.shape[0]):
        _lib.check(env.lib.fm_formation_step(env._h, actions[t].data_ptr(), C.byref(_keep_outputs(out, keep)), stream))
        rec.append({k: out[k].cpu().numpy().copy() for k in keep})
    vec = env.read_stats().cpu().numpy() if stats else None
    state = {k: v.clone() for k, v in env.get_state().items()}
    env.close()
    return vec, rec, state


def _host_stats(rec, N):
    """The statistics vector recomputed in float64 on the host from the device's own per-step outputs, and the sums of
    absolute values (the scale of the rounding error of a reordered sum)."""
    K = 15 * N + 2
    v, a = np.zeros(K), np.zeros(K)
    for r in rec:
        rew = r["reward"].astype(np.float64)
        v[:N] += rew.sum(0); a[:N] += np.abs(rew).sum(0)
        fin = r["done"].astype(bool).all(1)
        info = r["info"][fin].astype(np.float64).reshape(-1, N * 14)
        v[N:15 * N] += info.sum(0); a[N:15 * N] += np.abs(info).sum(0)
        v[15 * N] += fin.sum(); v[15 * N + 1] += len(fin)
    return v, a


def _assert_stats_match(vec, ref, scale, N):
    assert np.isfinite(vec).all()
    assert (vec[15 * N:] == ref[15 * N:]).all(), (vec[15 * N:], ref[15 * N:])
    err = np.abs(vec[:15 * N] - ref[:15 * N])
    assert (err <= 1e-12 * np.maximum(scale[:15 * N], 1e-300)).all(), err.max()


def _seeking_actions(cfg, B, T, seed=7, env_offset=0):
    """[T,B,N] goal-seeking actions of one trajectory (the trajectory is deterministic: every run with these actions
    sees the same states), so that agents latch and envs finish early."""
    import torch
    import fair_marl_b200 as fm
    env = fm.B200FormationVecEnv(cfg, num_envs=B, seed=seed, env_offset=env_offset)
    env.reset_tensor()
    rng, acts = np.random.default_rng(1), []
    for t in range(T):
        acts.append(_actions(_goal_seeking(_from_device(env.get_state()), rng)))
        env.step_tensor(acts[-1])
    env.close()
    return torch.stack(acts)


STATS_CASES = {
    "split": dict(N=3, O=3, B=70), "split_aligned": dict(N=3, O=2, B=64), "fused": dict(N=5, O=2, B=45),
    "walls": dict(N=3, O=2, B=45, num_walls=2), "collaborative": dict(N=4, O=2, B=37, collaborative=True),
    "info_every_step_0": dict(N=3, O=3, B=45, info_every_step=False), "auto_reset_0": dict(N=3, O=1, B=45, auto_reset=False),
    "optimal": dict(N=3, O=3, B=33, assignment="optimal", fairness_reward=False),
}


@pytest.mark.parametrize("case", sorted(STATS_CASES))
def test_episode_stats_match_host_sums(case):
    """fm_formation_stats_read against float64 sums, on the host, of the device's own per-step outputs (rewards of every
    env-step; info rows of the envs whose agents are all done), relative 1e-12, episode and env-step counts exact.  Without a
    caller info array, and with partial outputs, the vector is the same bit for bit; read(clear) zeroes the sums."""
    import torch
    import fair_marl_b200 as fm
    kw = dict(STATS_CASES[case])
    N, O, B = kw.pop("N"), kw.pop("O"), kw.pop("B")
    cfg = fm.FormationSimConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=9, **kw)
    T = 24
    acts = _seeking_actions(cfg, B, T)
    vec, rec, _ = _stats_run(cfg, B, acts)
    ref, scale = _host_stats(rec, N)
    _assert_stats_match(vec, ref, scale, N)
    assert vec[15 * N] > 0 and vec[15 * N + 1] == T * B
    if cfg.auto_reset:
        early = sum(int((r["done"].astype(bool).all(1)).sum()) for r in rec)
        assert early >= B                                              # time-outs at least
    for keep in [("obs", "node_obs", "adj", "reward", "done"), ("obs",), ("node_obs", "adj"), ("done",), ("reward", "info")]:
        got, _, _ = _stats_run(cfg, B, acts, keep=keep)
        assert (got == vec).all(), keep
    # clear: the next read sees only the steps after it
    env = fm.B200FormationVecEnv(cfg, num_envs=B, seed=7, episode_stats=True)
    env.reset_tensor()
    for t in range(T):
        env.step_tensor(acts[t])
    assert torch.equal(env.read_stats(clear=True).cpu(), torch.as_tensor(vec))
    assert (env.read_stats().cpu() == 0).all()
    env.step_tensor(acts[0])
    assert env.read_stats()[15 * N + 1].item() == B
    env.close()


def test_episode_stats_match_oracle():
    """Once against the float64 oracle stepped along from the device's own pre-step states: reward and info sums at the
    parity tolerance (the fairness ratios at theirs), counts exact."""
    import fair_marl_b200 as fm
    N, O, B, T = 3, 3, 48, 30
    cfg = FormationConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=12)
    env = fm.B200FormationVecEnv(_sim(cfg), num_envs=B, seed=7, episode_stats=True)
    orc = FormationOracle(cfg, B, seed=7)
    env.reset_tensor(); orc.reset()
    rng = np.random.default_rng(5)
    rew, info, eps = np.zeros(N), np.zeros((N, 14)), 0
    for t in range(T):
        cur = _from_device(env.get_state())
        orc.set_state(cur)
        a = _goal_seeking(cur, rng)
        env.step_tensor(_actions(a))
        ref = orc.step(a, autoreset=True)
        rew += ref["reward"].sum(0)
        fin = ref["done"].all(1)
        eps += int(fin.sum())
        for k, key in enumerate(INFO_KEYS):
            info[:, k] += ref["info"][key][fin].sum(0)
    vec = env.read_stats().cpu().numpy()
    assert vec[15 * N] == eps > B and vec[15 * N + 1] == T * B
    assert_close(vec[:N], rew, "reward sums")
    got = vec[N:15 * N].reshape(N, 14)
    for k, key in enumerate(INFO_KEYS):
        (assert_fairness_close if key in RATIO_KEYS else assert_close)(got[:, k], info[:, k], key)
    env.close()


def test_episode_stats_are_invisible():
    """With statistics on, every output and the state are the bytes of a run with them off (split and fused paths)."""
    import torch
    import fair_marl_b200 as fm
    for N, O, B in ((3, 3, 70), (5, 2, 45)):
        cfg = fm.FormationSimConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=9)
        acts = _seeking_actions(cfg, B, 20)
        on, off = _stats_run(cfg, B, acts, stats=True), _stats_run(cfg, B, acts, stats=False)
        for t, (a, b) in enumerate(zip(on[1], off[1])):
            for k in a:
                assert (a[k] == b[k]).all(), (N, t, k)
        for k in on[2]:
            assert torch.equal(on[2][k], off[2][k]), (N, k)
        partial_on, partial_off = _stats_run(cfg, B, acts, keep=("obs",)), _stats_run(cfg, B, acts, keep=("obs",), stats=False)
        for k in partial_on[2]:
            assert torch.equal(partial_on[2][k], partial_off[2][k]), (N, k)


def _stats_session(N, O, mode):
    """reset + 12 random-action steps at B = 4096 + 45 (two env-range lanes possible, ragged last tile), episode_length 4;
    `mode`: 'step' (single steps), 'many' (one fm_formation_step_many) or 'graph' (step_many captured, replayed once)."""
    import torch
    import fair_marl_b200 as fm
    B, T = 4096 + 45, 12
    cfg = fm.FormationSimConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=4,
                                info_every_step=False)
    g = torch.Generator(device="cuda").manual_seed(3)
    acts = torch.randint(0, 5, (T, B, N), generator=g, device="cuda", dtype=torch.int32)
    env = fm.B200FormationVecEnv(cfg, num_envs=B, seed=2, num_slots=T, episode_stats=True)
    env.reset_tensor()
    if mode == "step":
        for t in range(T):
            env.step_tensor(acts[t])
    elif mode == "many":
        env.rollout_tensor(acts)
    else:
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            env.rollout_tensor(acts)
        assert (env.read_stats().cpu() == 0).all()                  # capture does not execute
        graph.replay()
    vec = env.read_stats().cpu()
    torch.cuda.synchronize()
    env.close()
    return vec


@pytest.mark.parametrize("N,O", [(3, 3), (5, 2)])
def test_episode_stats_deterministic_across_launch_variants(N, O, monkeypatch):
    """The vector is the same bit for bit on every run and under every launch variant: PDL off, prefetch off, the fused
    kernel, two env-range lanes of step_many, a captured-graph replay."""
    import torch
    for k in FORM_SWITCHES:
        monkeypatch.delenv(k, raising=False)
    ref = _stats_session(N, O, "step")
    assert ref[15 * N] > 0 and (ref[N:15 * N] != 0).any()
    variants = [({}, "step"), ({}, "many"), ({"FM_FORM_PDL": "0"}, "step"), ({"FM_FORM_PREFETCH": "0"}, "step"),
                ({"FM_FORM_FUSED": "1"}, "step"), ({"FM_FORM_LANES": "2"}, "many"), ({}, "graph")]
    for switches, mode in variants:
        for k in FORM_SWITCHES:
            monkeypatch.delenv(k, raising=False)
        for k, v in switches.items():
            monkeypatch.setenv(k, v)
        got = _stats_session(N, O, mode)
        assert torch.equal(got, ref), (switches, mode)


def test_episode_stats_of_shards_add_up():
    """Two handles over env ranges [0, 64) and [64, 109) (env_offset) add up to one handle over [0, 109): counts exact, sums
    at 1e-12 -- what EpisodeStats all-reduces across ranks."""
    import torch
    import fair_marl_b200 as fm
    N = 3
    cfg = fm.FormationSimConfig(num_agents=N, num_obstacles=3, goal_rew=30.0, collision_rew=30.0, episode_length=5)
    g = torch.Generator(device="cuda").manual_seed(9)
    acts = torch.randint(0, 5, (15, 109, N), generator=g, device="cuda", dtype=torch.int32)
    whole, rec, _ = _stats_run(cfg, 109, acts)
    lo, _, _ = _stats_run(cfg, 64, acts[:, :64].contiguous())
    hi, _, _ = _stats_run(cfg, 45, acts[:, 64:].contiguous(), env_offset=64)
    _, scale = _host_stats(rec, N)
    _assert_stats_match(lo + hi, whole, scale, N)
    assert whole[15 * N] > 0


def test_make_train_env_gives_formation_env_with_stats():
    import types
    import torch
    import fair_marl_b200 as fm
    from fair_marl_b200.sharding import EpisodeStats
    args = types.SimpleNamespace(env_name="GraphMPE", scenario_name="nav_base_formation_graph_mask", n_rollout_threads=50,
                                 seed=3, num_agents=3, num_landmarks=3, num_obstacles=2, episode_length=6)
    env = fm.make_train_env(args, rank=1, world_size=2)
    assert isinstance(env, fm.B200FormationVecEnv) and env.num_envs == 25
    assert env.cfg.assignment == "optimal" and not env.cfg.fairness_reward
    env.reset_tensor()
    for t in range(6):
        env.step_tensor(torch.zeros(25, 3, dtype=torch.int32, device=env.device))
    st = EpisodeStats(3, device=env.device)
    st.all_reduce_async(env.read_stats())
    s = st.summary()
    assert s["episodes"] == 25 and s["env_steps"] == 150
    env.close()


@pytest.mark.reference
@pytest.mark.parametrize("variant", ["FA", "FA+FR", "OA", "RA"])
def test_shipped_actors_reach_goals_through_the_device_collector(variant):
    """The four shipped actors (model_weights/*/actor.pt), driven through RolloutCollector on the device, latch goals at
    5x or more the rate of random moves (the device twin of tests/test_formation_closed_loop.py)."""
    import os
    import torch
    import fair_marl_b200 as fm
    from fair_marl_b200.policy import config_from_state_dict, load_reference_state_dict
    from oracle import reference_shim
    mode, fair = {"FA+FR": ("fair", True), "FA": ("fair", False), "OA": ("optimal", False), "RA": ("random", False)}[variant]
    N, B, L = 3, 16, 25
    cfg = fm.FormationSimConfig(num_agents=N, num_obstacles=3, goal_rew=30.0, collision_rew=30.0, assignment=mode,
                                fairness_reward=fair, episode_length=L)

    def latches(dones):
        """Agent done onsets before the time-out, counted with a host step counter per env ([S,B,N] uint8)."""
        d = dones.bool().cpu().numpy()
        step, prev, n = np.zeros(B, int), np.zeros((B, N), bool), 0
        for t in range(d.shape[0]):
            step += 1
            n += int((d[t] & ~prev)[step < L].sum())
            fin = d[t].all(1)
            prev = d[t] & ~fin[:, None]
            step[fin] = 0
        return n

    sd = torch.load(os.path.join(reference_shim.REFERENCE_ROOT, "model_weights", variant, "actor.pt"), map_location="cpu",
                    weights_only=False)
    pc = config_from_state_dict(sd)
    env = fm.B200FormationVecEnv(cfg, num_envs=B, seed=3)
    actor = fm.DenseGraphActor(pc).to(env.device).eval()
    load_reference_state_dict(actor, sd)
    actor = actor.to(env.device)
    critic = fm.DenseGraphCritic(pc).to(env.device).eval()
    col = fm.RolloutCollector(env, actor, critic, deterministic=True)
    col.warmup()
    dones = []
    for _ in range(2):
        col.run()
        dones.append(col.buffer.dones.clone())
        col.buffer.after_update()
    n_policy = latches(torch.cat(dones))
    env2 = fm.B200FormationVecEnv(cfg, num_envs=B, seed=3)
    env2.reset_tensor()
    g = torch.Generator(device="cuda").manual_seed(3)
    rnd = [env2.step_tensor(torch.randint(0, 5, (B, N), generator=g, device="cuda", dtype=torch.int32))["done"].clone()
           for _ in range(2 * L)]
    n_random = latches(torch.stack(rnd).to(torch.uint8))
    assert n_policy >= 20 and n_policy >= 5 * max(n_random, 1), (variant, n_policy, n_random)
    env.close(); env2.close()
