"""The optimal-assignment formation scenario (OA, nav_base_formation_graph_mask.py) at 6 and 7 agents, on the GPU.  Its
min-sum matching is f_min_sum_sap (scipy's shortest augmenting path, csrc/fm_form.cuh), run at every reset and in agent 0's
reward call on every step.  Helpers and the oracle plumbing are those of tests/test_gpu_formation.py."""
from dataclasses import fields

import numpy as np
import pytest

from oracle.formation import FormationConfig, FormationOracle, FormationState
from parity_util import assert_close
from test_gpu_formation import (FORM_SWITCHES, INT_FIELDS, LAUNCH_VARIANTS, SHORT, _actions, _case, _from_device, _goal_seeking,
                                _np, _rollout_matches_oracle, _scripted_session, _sim, _walls_from_device)

pytestmark = pytest.mark.gpu

OA_CASES = [
    _case(6, 0, 45, False, False, "optimal", 0, early=True), _case(7, 0, 45, False, False, "optimal", 0, early=True),
    _case(6, 3, 17, False, False, "optimal", 0, **SHORT), _case(7, 3, 1, False, False, "optimal", 0, **SHORT),
    _case(6, 8, 1, True, False, "optimal", 0, **SHORT), _case(7, 8, 17, False, False, "optimal", 0, **SHORT),
    _case(6, 2, 17, False, False, "optimal", 1, **SHORT), _case(7, 1, 45, True, False, "optimal", 2, **SHORT),   # walls
    _case(6, 3, 45, False, False, "optimal", 0, "vmax_none", max_speed=None, **SHORT),
    _case(7, 3, 17, False, False, "optimal", 0, "vmax_0.7", max_speed=0.7, **SHORT),
]


@pytest.mark.parametrize("N,O,B,collab,fair,assignment,W,opts", OA_CASES)
def test_oa_reset_and_rollout_match_oracle(N, O, B, collab, fair, assignment, W, opts):
    """Reset bit for bit against the oracle (goal_match is scipy's col_ind of the reset distances), then a goal-seeking
    rollout across auto-resets, every step's outputs and state within the parity tolerance, goal_match exact."""
    cfg = FormationConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0,
                          episode_length=opts.get("episode_length", 15), max_speed=opts.get("max_speed", 2.0),
                          collaborative=collab, fairness_reward=fair, assignment=assignment, num_walls=W)
    _rollout_matches_oracle(cfg, B, opts.get("steps", 32), opts.get("early", False))


def test_oa_masked_reset_matches_oracle():
    """reset(mask) in mid-episode at N = 7: the masked envs draw a new episode and solve the min-sum matching of its
    distances (bit for bit), the others are re-observed."""
    import fair_marl_b200 as fm
    N, O, B = 7, 2, 45
    cfg = FormationConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=20,
                          fairness_reward=False, assignment="optimal")
    env = fm.B200FormationVecEnv(_sim(cfg), num_envs=B, seed=21, env_offset=2)
    orc = FormationOracle(cfg, B, seed=21, env_offset=2)
    env.reset_tensor()
    rng = np.random.default_rng(8)
    for t in range(5):
        env.step_tensor(_actions(_goal_seeking(_from_device(env.get_state()), rng)))
    dev = env.get_state()
    pre = _from_device(dev)
    orc.set_state(pre)
    _walls_from_device(orc, dev)
    mask = rng.random(B) < 0.4
    mask[:2] = (True, False)
    out, ref = _np(env.reset_tensor(mask.astype(np.uint8))), orc.reset(mask)
    post, rpost = _from_device(env.get_state()), orc.get_state()
    for f in ("pos", "landmark_pos", "obstacle_pos", "goal_match"):
        assert (getattr(post, f)[mask] == getattr(rpost, f)[mask]).all(), f
        assert (getattr(post, f)[~mask] == getattr(pre, f)[~mask]).all(), f
    for f in ("goal_match", "step", "episode", "status"):
        assert (getattr(post, f) == getattr(rpost, f)).all(), f
    assert_close(out["obs"], ref["obs"], "obs")
    assert_close(out["node_obs"], ref["node_obs"], "node_obs")
    assert_close(out["adj_env"], ref["adj"], "adj")
    for f in fields(FormationState):
        if f.name not in INT_FIELDS and f.name != "status":
            assert_close(getattr(post, f.name), getattr(rpost, f.name), f.name)
    env.close()


# _scripted_session picks the assignment from (N + O) % 3: these shapes are OA
@pytest.mark.parametrize("N,O", [(6, 1), (7, 0)])
def test_oa_launch_variants_are_bitwise_identical(N, O, monkeypatch):
    """The default, PDL off, prefetch off, both off and FM_FORM_FUSED=1 give the same bytes in a scripted session with
    resets on every step, a masked reset, one- and two-lane rollouts and a captured CUDA graph replayed twice."""
    import torch
    assert ("fair", "optimal", "random")[(N + O) % 3] == "optimal"
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


def test_oa_collector_episode_with_stats_replays_bitwise():
    """A RolloutCollector episode at N = 7 OA with episode statistics on; replaying its actions through a second env gives
    every slab bit for bit, and the same statistics vector."""
    import torch
    import fair_marl_b200 as fm
    N, O, B = 7, 1, 64
    cfg = fm.FormationSimConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, assignment="optimal",
                                fairness_reward=False)
    env = fm.B200FormationVecEnv(cfg, num_envs=B, seed=5, episode_stats=True)
    pc = fm.PolicyConfig(num_agents=N, obs_dim=11, node_feat_dim=13)
    torch.manual_seed(0)
    actor, critic = fm.DenseGraphActor(pc).to(env.device).eval(), fm.DenseGraphCritic(pc).to(env.device).eval()
    with torch.no_grad():
        actor.action_out.weight.mul_(100.0)
    col = fm.RolloutCollector(env, actor, critic, deterministic=True)
    buf = col.buffer
    col.warmup(); col.run()
    torch.cuda.synchronize()
    env2 = fm.B200FormationVecEnv(cfg, num_envs=B, seed=5, episode_stats=True)
    r = env2.reset_tensor()
    assert torch.equal(r["obs"], buf.obs[0]) and torch.equal(r["node_obs"], buf.node_obs[0])
    for t in range(cfg.episode_length):
        o = env2.step_tensor(buf.actions_env[t])
        assert torch.equal(o["obs"], buf.obs[t + 1]), t
        assert torch.equal(o["node_obs"], buf.node_obs[t + 1]), t
        assert torch.equal(o["adj_env"], buf.adj_env[t + 1]), t
        assert torch.equal(o["reward"], buf.rewards[t, :, :, 0]), t
        assert torch.equal(o["done"], buf.dones[t].bool()), t
    s1, s2 = env.read_stats(), env2.read_stats()
    assert torch.equal(s1, s2)
    assert s1[15 * N].item() >= B and s1[15 * N + 1].item() == cfg.episode_length * B
    env.close(); env2.close()
