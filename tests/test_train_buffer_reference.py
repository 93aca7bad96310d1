"""``-m "gpu and reference"``: oracle/graph_buffer.py and the device buffer's returns and generators against the live
reference ``GraphReplayBuffer`` and ``ValueNorm`` (onpolicy/utils/graph_buffer.py, valuenorm.py).  The generators'
permutation is fed to the reference through ``torch.randperm``.  Skips where there is no reference checkout
(FAIRMARL_REFERENCE_ROOT)."""
from argparse import Namespace

import numpy as np
import pytest
import torch

from oracle import graph_buffer as ogb

pytestmark = [pytest.mark.gpu, pytest.mark.reference]


def _live(T, B, N, E, gae, proper, norm):
    from oracle import reference_shim
    reference_shim.install_stubs()
    import gym
    from onpolicy.utils.graph_buffer import GraphReplayBuffer
    Box, Disc = gym.spaces.Box, gym.spaces.Discrete
    args = Namespace(episode_length=T, n_rollout_threads=B, hidden_size=64, recurrent_N=1, gamma=0.99, gae_lambda=0.95,
                     use_gae=gae, use_popart=False, use_valuenorm=norm, use_proper_time_limits=proper, use_centralized_V=True)
    return GraphReplayBuffer(args, N, Box(0, 0, (7,)), Box(0, 0, (7 * N,)), Box(0, 0, (E, 11)), Box(0, 0, (1,)), Box(0, 0, (N,)),
                             Box(0, 0, (E, E)), Disc(5))


def _device_buffer(T, B, N, E, gae, proper, seed):
    from fair_marl_b200.rollout import DeviceRolloutBuffer
    b = DeviceRolloutBuffer(T, B, N, E, device="cuda", use_gae=gae, use_proper_time_limits=proper)
    g = torch.Generator(device="cuda").manual_seed(seed)
    for name in ("obs", "node_obs", "adj_env", "rnn_states", "rnn_states_critic", "action_log_probs", "value_preds", "rewards", "returns"):
        x = getattr(b, name)
        x.copy_(torch.randn(x.shape, device="cuda", generator=g))
    b.actions.copy_(torch.randint(0, 5, b.actions.shape, device="cuda", generator=g).float())
    for name in ("masks", "bad_masks", "active_masks"):
        getattr(b, name).copy_((torch.rand(b.masks.shape, device="cuda", generator=g) > 0.2).float())
    return b


def _fill(ref, b):
    for name in ("share_obs", "obs", "node_obs", "adj", "agent_id", "share_agent_id", "rnn_states", "rnn_states_critic", "actions",
                 "available_actions", "value_preds", "returns", "masks", "bad_masks", "active_masks", "action_log_probs", "rewards"):
        getattr(ref, name)[...] = getattr(b, name).cpu().numpy()


def _value_norm():
    from onpolicy.utils.valuenorm import ValueNorm
    vn = ValueNorm(1, device=torch.device("cuda"))
    for s in range(3):
        vn.update(7.5 + 3.0 * torch.randn(64, 1, generator=torch.Generator().manual_seed(s)))
    return vn


@pytest.mark.parametrize("gae,proper,norm", [(g, p, n) for g in (True, False) for p in (False, True) for n in (False, True)])
def test_returns_match_the_live_reference(gae, proper, norm):
    T, B, N, E = 25, 16, 3, 9
    b = _device_buffer(T, B, N, E, gae, proper, seed=1)
    ref = _live(T, B, N, E, gae, proper, norm)
    _fill(ref, b)
    vn = _value_norm() if norm else None
    nv = torch.randn(B * N, 1, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    slabs = {k: getattr(ref, k).copy() for k in ("value_preds", "rewards", "masks", "bad_masks", "returns")}
    ref.compute_returns(nv.cpu().numpy().reshape(B, N, 1), vn)
    b.compute_returns(nv, vn)
    assert np.array_equal(b.returns.cpu().numpy(), ref.returns)
    if vn is None:                                      # the oracle restates the live loop (its ValueNorm is numpy)
        ogb.compute_returns(slabs, nv.cpu().numpy().reshape(B, N, 1), None, use_gae=gae, use_proper_time_limits=proper)
        assert np.array_equal(slabs["returns"], ref.returns)


@pytest.mark.parametrize("mode,K,L", [("feed_forward", 4, 0), ("recurrent", 3, 10), ("naive_recurrent", 4, 0)])
def test_generators_match_the_live_reference(mode, K, L, monkeypatch):
    T, B, N, E = 25, 16, 3, 9
    b = _device_buffer(T, B, N, E, True, False, seed=3)
    ref = _live(T, B, N, E, True, False, False)
    _fill(ref, b)
    adv = b.advantages()
    g = torch.Generator(device="cuda").manual_seed(7)
    dev = {"feed_forward": lambda: b.feed_forward_generator(adv, K, generator=g),
           "recurrent": lambda: b.recurrent_generator(adv, K, L, generator=g),
           "naive_recurrent": lambda: b.naive_recurrent_generator(adv, K, generator=g)}[mode]
    units = {"feed_forward": T * B * N, "recurrent": T * B * N // max(L, 1), "naive_recurrent": B * N}[mode]
    perm = torch.randperm(units, device="cuda", generator=torch.Generator(device="cuda").manual_seed(7)).cpu()
    monkeypatch.setattr(torch, "randperm", lambda n, *a, **k: perm.clone())
    a = adv.cpu().numpy()
    live = {"feed_forward": lambda: ref.feed_forward_generator(a, K),
            "recurrent": lambda: ref.recurrent_generator(a, K, L),
            "naive_recurrent": lambda: ref.naive_recurrent_generator(a, K)}[mode]
    want = list(live())
    monkeypatch.undo()
    got = list(dev())
    assert len(got) == len(want)
    for gb, wb in zip(got, want):
        for x, y in zip(gb, wb):
            y = np.asarray(y)
            assert np.array_equal(x.cpu().numpy().reshape(y.shape), y.astype(x.cpu().numpy().dtype))
