"""DeviceRolloutBuffer (plain torch, here on the CPU device) vs the reference's GraphReplayBuffer fed through the
reference's GMPERunner.insert logic (graph_mpe_runner.py:438-488, restated below line by line because GMPERunner
itself needs a trainer / tensorboard).  Needs the original project's checkout (FAIRMARL_REFERENCE_ROOT)."""
from argparse import Namespace

import numpy as np
import pytest
import torch

from fair_marl_b200.rollout import DeviceRolloutBuffer
from oracle import reference_shim

pytestmark = pytest.mark.reference


def _reference_buffer(T, B, N, E, H):
    reference_shim.install_stubs()
    import gym
    from onpolicy.utils.graph_buffer import GraphReplayBuffer
    Box, Disc = gym.spaces.Box, gym.spaces.Discrete
    args = Namespace(episode_length=T, n_rollout_threads=B, hidden_size=H, recurrent_N=1, gamma=0.99, gae_lambda=0.95,
                     use_gae=True, use_popart=False, use_valuenorm=False, use_proper_time_limits=False, use_centralized_V=True)
    return GraphReplayBuffer(args, N, Box(0, 0, (7,)), Box(0, 0, (7 * N,)), Box(0, 0, (E, 11)), Box(0, 0, (1,)), Box(0, 0, (N,)),
                             Box(0, 0, (E, E)), Disc(5))


def _runner_insert(buf, B, N, H, obs, agent_id, node_obs, adj, rewards, dones, values, actions, logp, rnn, rnn_c):
    """GMPERunner.insert, graph_mpe_runner.py:438-488 (use_centralized_V branch)."""
    dones_env = np.all(dones, axis=1)
    rnn[dones] = np.zeros((dones.sum(), 1, H), dtype=np.float32)
    rnn_c[dones] = np.zeros((dones.sum(), 1, H), dtype=np.float32)
    masks = np.ones((B, N, 1), dtype=np.float32)
    masks[dones] = np.zeros((dones.sum(), 1), dtype=np.float32)
    active = np.ones((B, N, 1), dtype=np.float32)
    active[dones] = np.zeros((dones.astype(int).sum(), 1), dtype=np.float32)
    active[dones_env] = np.ones((dones_env.astype(int).sum(), N, 1), dtype=np.float32)
    share_obs = np.expand_dims(obs.reshape(B, -1), 1).repeat(N, axis=1)
    share_id = np.expand_dims(agent_id.reshape(B, -1), 1).repeat(N, axis=1)
    buf.insert(share_obs, obs, node_obs, adj, agent_id, share_id, rnn, rnn_c, actions, logp, values, rewards[:, :, None],
               masks, active_masks=active)


def test_buffer_matches_reference_insert_and_returns():
    T, B, N, O, H = 6, 5, 3, 2, 8
    E = 2 * N + O
    rng = np.random.default_rng(0)
    ref = _reference_buffer(T, B, N, E, H)
    dev = DeviceRolloutBuffer(T, B, N, E, hidden_size=H, device="cpu")
    agent_id = np.tile(np.arange(N)[None, :, None], (B, 1, 1))

    def obs_set():
        adj_env = rng.random((B, E, E)).astype(np.float32)
        return (rng.normal(size=(B, N, 7)).astype(np.float32), rng.normal(size=(B, N, E, 11)).astype(np.float32), adj_env)

    o0, n0, a0 = obs_set()                                   # GMPERunner.warmup (:198-203)
    ref.obs[0], ref.node_obs[0], ref.adj[0], ref.agent_id[0] = o0, n0, np.repeat(a0[:, None], N, 1), agent_id
    ref.share_obs[0] = np.expand_dims(o0.reshape(B, -1), 1).repeat(N, axis=1)
    ref.share_agent_id[0] = np.expand_dims(agent_id.reshape(B, -1), 1).repeat(N, axis=1)
    v0 = dev.env_views(0, with_step=False)
    v0["obs"].copy_(torch.as_tensor(o0)); v0["node_obs"].copy_(torch.as_tensor(n0)); v0["adj"].copy_(torch.as_tensor(a0))
    for t in range(T):
        o, n, a = obs_set()
        rew = rng.normal(size=(B, N)).astype(np.float32)
        dones = np.zeros((B, N), bool)
        if t == 3:
            dones[:] = True                                  # all agents of every env finish together (episode end)
        if t == 4:
            dones[1, 0] = True                               # a single agent done (formation family): active_masks path
        vals, acts = rng.normal(size=(B, N, 1)).astype(np.float32), rng.integers(0, 5, (B, N, 1)).astype(np.float32)
        logp = rng.normal(size=(B, N, 1)).astype(np.float32)
        rnn, rnn_c = rng.normal(size=(B, N, 1, H)).astype(np.float32), rng.normal(size=(B, N, 1, H)).astype(np.float32)
        # device path: the "kernel" writes slab t + 1 in place, then the policy-side insert
        v = dev.env_views(t + 1)
        v["obs"].copy_(torch.as_tensor(o)); v["node_obs"].copy_(torch.as_tensor(n)); v["adj"].copy_(torch.as_tensor(a))
        v["reward"].copy_(torch.as_tensor(rew)); v["done"].copy_(torch.as_tensor(dones.astype(np.uint8)))
        dev.insert_policy(torch.as_tensor(rnn.reshape(B * N, 1, H)), torch.as_tensor(rnn_c.reshape(B * N, 1, H)),
                          torch.as_tensor(acts.reshape(B * N, 1)), torch.as_tensor(logp.reshape(B * N, 1)),
                          torch.as_tensor(vals.reshape(B * N, 1)))
        _runner_insert(ref, B, N, H, o, agent_id, n, np.repeat(a[:, None], N, 1), rew, dones, vals, acts, logp, rnn.copy(), rnn_c.copy())
    nv = rng.normal(size=(B, N, 1)).astype(np.float32)
    ref.compute_returns(nv)
    dev.compute_returns(torch.as_tensor(nv))
    for name in ("obs", "node_obs", "adj", "share_obs", "agent_id", "share_agent_id", "rnn_states", "rnn_states_critic", "actions",
                 "action_log_probs", "value_preds", "rewards", "masks", "active_masks", "bad_masks", "available_actions"):
        got, want = getattr(dev, name).numpy(), getattr(ref, name)
        assert got.shape == want.shape, (name, got.shape, want.shape)
        assert np.array_equal(got, want), name
    assert np.allclose(dev.returns.numpy(), ref.returns, rtol=1e-6, atol=1e-6)
    assert dev.step == ref.step
    ref.after_update(); dev.after_update()
    for name in ("obs", "node_obs", "adj", "share_obs", "rnn_states", "masks", "active_masks"):
        assert np.array_equal(getattr(dev, name).numpy()[0], getattr(ref, name)[0]), name
