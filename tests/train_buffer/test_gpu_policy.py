"""The trainer's input on the device rollout buffer (csrc/fm_buffer.cu behind DeviceRolloutBuffer):

* the returns scan (fm_buffer_returns) bit for bit oracle/graph_buffer.py in all 8 (GAE x proper time limits x value
  normaliser) combinations at (T, B, N) = (25, 65 536, 3), (25, 4 096, 16), (7, 1, 1) and a ragged shape; bit for bit the
  torch loop compute_returns ran on a CUDA buffer before it became a kernel; a captured compute_returns + advantages
  replays to the same bits;
* the advantages (fm_buffer_advantages): mean and std within one float32 ulp of float32(float64 truth), the normalised
  values bit for bit GR_MAPPO.train's formula applied to the device's mean and std, NaN when nothing is active, two runs
  identical;
* the three generators (fm_buffer_minibatch): every field of every mini-batch of an epoch bit for bit the oracle's
  restatement given the permutation drawn from the same seeded generator, at several (num_mini_batch, L), with
  T % L != 0 and mini_batch_size, for navigation (E = 9 and 35) and formation shapes; the union of an epoch's samples is
  the expected set, the remainder dropped as the reference drops it;
* RolloutCollector end to end at navigation N = 3 and formation N = 5: finish(value_normalizer) equals the oracle run on
  the buffer's own slabs, and every mini-batch feeds DenseGraphActor / DenseGraphCritic forward and backward.
"""
import numpy as np
import pytest
import torch

from oracle import graph_buffer as ogb
from test_train_buffer_cpu import COMBOS, TorchNorm as _TorchNorm, oracle_slabs, random_buffer, trained_value_norm

pytestmark = pytest.mark.gpu


def TorchNorm(vn):
    return _TorchNorm(vn, "cuda")                     # the reference's normaliser lives on the training device


RETURN_SHAPES = [(25, 65536, 3), (25, 4096, 16), (7, 1, 1), (13, 333, 5)]


def _vn(norm):
    return trained_value_norm() if norm else None


@pytest.mark.parametrize("gae,proper,norm", COMBOS)
@pytest.mark.parametrize("shape", RETURN_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_returns_kernel_matches_the_oracle_bit_for_bit(shape, gae, proper, norm):
    T, B, N = shape
    rng = np.random.default_rng(T * B + N)
    b = random_buffer(T, B, N, rng, device="cuda", use_gae=gae, use_proper_time_limits=proper)
    nv = torch.as_tensor(rng.standard_normal((B * N, 1)).astype(np.float32)).cuda()
    vn = _vn(norm)
    ref = oracle_slabs(b)
    ogb.compute_returns(ref, nv.cpu().numpy().reshape(B, N, 1), vn, use_gae=gae, use_proper_time_limits=proper)
    b.compute_returns(nv, TorchNorm(vn) if norm else None)
    assert np.array_equal(b.returns.cpu().numpy(), ref["returns"])
    assert np.array_equal(b.value_preds.cpu().numpy(), ref["value_preds"])


@pytest.mark.parametrize("shape", RETURN_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_returns_kernel_is_the_previous_torch_loop(shape):
    """compute_returns on a CUDA buffer ran this loop (GAE, no normaliser, no proper time limits); the kernel gives the
    same bits."""
    T, B, N = shape
    rng = np.random.default_rng(5)
    b = random_buffer(T, B, N, rng, device="cuda")
    nv = torch.as_tensor(rng.standard_normal((B * N, 1)).astype(np.float32)).cuda()
    v, r, m = b.value_preds.clone(), b.rewards.clone(), b.masks.clone()
    v[-1] = nv.view_as(v[-1])
    ret = b.returns.clone()
    gae = torch.zeros_like(v[0])
    for t in reversed(range(T)):
        delta = r[t] + b.gamma * v[t + 1] * m[t + 1] - v[t]
        gae = delta + b.gamma * b.gae_lambda * m[t + 1] * gae
        ret[t] = gae + v[t]
    b.compute_returns(nv)
    assert torch.equal(b.returns, ret) and torch.equal(b.value_preds, v)


def test_captured_returns_and_advantages_replay_to_the_same_bits():
    T, B, N = 25, 4096, 3
    rng = np.random.default_rng(9)
    b = random_buffer(T, B, N, rng, device="cuda")
    vn = TorchNorm(trained_value_norm())
    nv = torch.as_tensor(rng.standard_normal((B * N, 1)).astype(np.float32)).cuda()
    slabs0 = b.value_preds.clone()
    b.compute_returns(nv, vn)
    eager_ret, eager_adv = b.returns.clone(), b.advantages(vn).clone()
    b.returns.zero_()
    b.value_preds.copy_(slabs0)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        b.compute_returns(nv, vn)
        adv = b.advantages(vn)
    b.returns.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(b.returns, eager_ret) and torch.equal(adv, eager_adv)


# ---- advantages ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("norm", [False, True])
@pytest.mark.parametrize("shape", [(25, 65536, 3), (25, 4096, 16), (7, 1, 1), (13, 333, 5)], ids=lambda s: "x".join(map(str, s)))
def test_advantages_statistics_and_normalisation(shape, norm):
    T, B, N = shape
    rng = np.random.default_rng(B + N)
    b = random_buffer(T, B, N, rng, device="cuda")
    b.active_masks[0].fill_(1.0)                                     # at least one active entry even at B = N = 1
    b.returns.copy_(torch.as_tensor((3.0 + 2.0 * rng.standard_normal((T + 1, B, N, 1))).astype(np.float32)))
    vn = _vn(norm)
    adv = b.advantages(TorchNorm(vn) if norm else None)
    mean, std = b.advantage_stats.cpu().numpy()
    buf = {k: getattr(b, k).cpu().numpy() for k in ("returns", "value_preds", "active_masks")}
    raw = ogb.raw_advantages(buf, vn)
    act = buf["active_masks"][:-1] != 0
    x = raw[act].astype(np.float64)
    m64 = x.mean()
    s64 = np.sqrt(((x - m64) ** 2).mean())
    for got, want in ((mean, m64), (std, s64)):
        w = np.float32(want)
        assert abs(got - w) <= np.spacing(abs(w)), (got, want)
    assert np.array_equal(adv.cpu().numpy(), ogb.normalise_advantages(raw, mean, std))
    again = b.advantages(TorchNorm(vn) if norm else None)
    assert torch.equal(adv, again) and torch.equal(b.advantage_stats.cpu(), torch.as_tensor([mean, std]))


def test_advantages_with_no_active_entry_are_nan():
    b = random_buffer(6, 10, 3, np.random.default_rng(1), device="cuda")
    b.active_masks.zero_()
    adv = b.advantages()
    assert torch.isnan(adv).all() and torch.isnan(b.advantage_stats).all()
    buf = {k: getattr(b, k).cpu().numpy() for k in ("returns", "value_preds", "active_masks")}
    want, mean, std = ogb.advantages(buf)
    assert np.isnan(mean) and np.isnan(std) and np.isnan(want).all()


# ---- generators ---------------------------------------------------------------------------------------------------------
def full_buffer(T, B, N, E, obs_dim, F, seed, ids=False):
    """A CUDA DeviceRolloutBuffer with every field random (value_preds = the sample's flat (t, b, n) index with ids)."""
    from fair_marl_b200.rollout import DeviceRolloutBuffer
    b = DeviceRolloutBuffer(T, B, N, E, obs_dim=obs_dim, node_feat_dim=F, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(seed)
    for name in ("obs", "node_obs", "adj_env", "rnn_states", "rnn_states_critic", "action_log_probs", "value_preds", "returns"):
        x = getattr(b, name)
        x.copy_(torch.randn(x.shape, device="cuda", generator=g))
    b.actions.copy_(torch.randint(0, 5, b.actions.shape, device="cuda", generator=g).float())
    b.masks.copy_((torch.rand(b.masks.shape, device="cuda", generator=g) > 0.2).float())
    b.active_masks.copy_((torch.rand(b.masks.shape, device="cuda", generator=g) > 0.2).float())
    if ids:
        b.value_preds[:T].copy_(torch.arange(T * B * N, device="cuda", dtype=torch.float32).view(T, B, N, 1))
    return b


def reference_layout(b):
    """The buffer as GraphReplayBuffer stores it (share_obs / share_agent_id / adj materialised per agent), numpy."""
    names = ("share_obs", "obs", "node_obs", "adj", "agent_id", "share_agent_id", "rnn_states", "rnn_states_critic", "actions",
             "available_actions", "value_preds", "returns", "masks", "active_masks", "action_log_probs", "rewards", "bad_masks")
    return {k: getattr(b, k).contiguous().cpu().numpy() for k in names}


def _draw(b, mode, K, mbs, L, seed, adv):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if mode == "feed_forward":
        return b.feed_forward_generator(adv, K, mbs, generator=g)
    if mode == "recurrent":
        return b.recurrent_generator(adv, K, L, generator=g)
    return b.naive_recurrent_generator(adv, K, generator=g)


def _units(b, mode, L):
    T, B, N = b.episode_length, b.n_rollout_threads, b.num_agents
    return {"feed_forward": T * B * N, "recurrent": T * B * N // max(L, 1), "naive_recurrent": B * N}[mode]


GEN_SHAPES = {"nav_E9": (25, 40, 3, 9, 7, 11), "form_N5": (25, 24, 5, 12, 11, 13), "nav_E35": (10, 6, 16, 35, 7, 11)}
GEN_CASES = [("feed_forward", 1, None, 0), ("feed_forward", 4, None, 0), ("feed_forward", 3, 100, 0),
             ("recurrent", 1, None, 10), ("recurrent", 4, None, 10), ("recurrent", 3, None, 7), ("recurrent", 5, None, 25),
             ("naive_recurrent", 1, None, 0), ("naive_recurrent", 2, None, 0), ("naive_recurrent", 6, None, 0)]


@pytest.mark.parametrize("mode,K,mbs,L", GEN_CASES, ids=lambda c: str(c))
@pytest.mark.parametrize("shape", list(GEN_SHAPES), ids=str)
def test_generators_match_the_oracle_bit_for_bit(shape, mode, K, mbs, L):
    T, B, N, E, D, F = GEN_SHAPES[shape]
    b = full_buffer(T, B, N, E, D, F, seed=3)
    adv = b.advantages()
    seed = 17 + K
    batches = list(_draw(b, mode, K, mbs, L, seed, adv))
    perm = torch.randperm(_units(b, mode, L), device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed)).cpu().numpy()
    ref, a = reference_layout(b), adv.cpu().numpy()
    if mode == "feed_forward":
        want = list(ogb.feed_forward_batches(ref, a, perm, K, mbs))
    elif mode == "recurrent":
        want = list(ogb.recurrent_batches(ref, a, perm, K, L))
    else:
        want = list(ogb.naive_recurrent_batches(ref, a, perm, K))
    assert len(batches) == len(want) == K
    for got, w in zip(batches, want):
        assert len(got) == len(w) == 16
        for name, x, y in zip(ogb.SAMPLE_FIELDS, got, w):
            assert x.is_cuda and tuple(x.shape) == y.shape, (name, tuple(x.shape), y.shape)
            assert np.array_equal(x.cpu().numpy(), y.astype(x.cpu().numpy().dtype)), name
            if name in ("agent_id", "share_agent_id"):
                assert x.dtype == torch.int32


@pytest.mark.parametrize("mode,K,mbs,L", [("feed_forward", 7, None, 0), ("feed_forward", 4, 333, 0), ("recurrent", 4, None, 10),
                                          ("recurrent", 6, None, 7), ("naive_recurrent", 4, None, 0)], ids=lambda c: str(c))
def test_epoch_covers_the_expected_samples(mode, K, mbs, L):
    """value_preds holds each sample's flat (t, b, n) index: the epoch's samples are perm[:K per] mapped back, each once;
    the remainder (T B N % (K per) samples, or the chunks' tail) is dropped as in the reference."""
    T, B, N = 25, 40, 3
    b = full_buffer(T, B, N, 9, 7, 11, seed=4, ids=True)
    adv = b.advantages()
    seed = 99
    got = torch.cat([mb[9][:, 0] for mb in _draw(b, mode, K, mbs, L, seed, adv)]).cpu().numpy().astype(np.int64)
    perm = torch.randperm(_units(b, mode, L), device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed)).cpu().numpy()
    if mode == "feed_forward":
        per = mbs or T * B * N // K
        want = perm[:K * per]
    elif mode == "recurrent":
        per = T * B * N // L // K
        f = (perm[:K * per, None] * L + np.arange(L)[None, :]).ravel()      # flat (b, n, t)
        t, bn = f % T, f // T
        want = t * B * N + bn
    else:
        want = np.arange(T * B * N)
    assert len(got) == len(set(got.tolist())) == len(want)
    assert np.array_equal(np.sort(got), np.sort(want))


# ---- the collector end to end -------------------------------------------------------------------------------------------
COLLECTOR_SHAPES = [("navigation", 3, 3), ("formation", 5, 2)]


def _collector(family, N, O, B=48, T=8):
    import fair_marl_b200 as fm
    import parity_util
    parity_util.MAPPING = "auto"
    f = {"navigation": (7, 11), "formation": (11, 13)}[family]
    if family == "navigation":
        from oracle.navgraph import NavConfig
        env = fm.B200GraphVecEnv(parity_util.sim_config_from(NavConfig(num_agents=N, num_obstacles=O, episode_length=T)),
                                 num_envs=B, seed=11)
    else:
        env = fm.B200FormationVecEnv(fm.FormationSimConfig(num_agents=N, num_obstacles=O, episode_length=T), num_envs=B, seed=11)
    torch.manual_seed(0)
    cfg = fm.PolicyConfig(num_agents=N, obs_dim=f[0], node_feat_dim=f[1])
    actor, critic = fm.DenseGraphActor(cfg).cuda(), fm.DenseGraphCritic(cfg).cuda()
    col = fm.RolloutCollector(env, actor, critic, generator=torch.Generator(device="cuda").manual_seed(5))
    col.warmup()
    col.run()
    return env, col, actor, critic


@pytest.mark.parametrize("shape", COLLECTOR_SHAPES, ids=lambda s: f"{s[0]}-N{s[1]}")
def test_collector_finish_advantages_and_ppo_shaped_consumer(shape):
    env, col, actor, critic = _collector(*shape)
    b = col.buffer
    vn = trained_value_norm(7)
    ref = oracle_slabs(b)
    col.finish(TorchNorm(vn))
    torch.cuda.synchronize()
    nv = b.value_preds[-1].cpu().numpy()                     # the critic's bootstrap value, stored by the kernel
    ogb.compute_returns(ref, nv, vn)
    assert np.array_equal(b.returns.cpu().numpy(), ref["returns"])
    adv = b.advantages(TorchNorm(vn))
    refb = {k: getattr(b, k).cpu().numpy() for k in ("returns", "value_preds", "active_masks")}
    raw = ogb.raw_advantages(refb, vn)
    mean, std = b.advantage_stats.cpu().numpy()
    assert np.array_equal(adv.cpu().numpy(), ogb.normalise_advantages(raw, mean, std))
    # ppo_update-shaped consumer: evaluate the mini-batch's actions and values with autograd, then a backward
    params = list(actor.parameters()) + list(critic.parameters())
    n = 0
    for sample in b.feed_forward_generator(adv, 4):
        (share_obs, obs, node_obs, adj, agent_id, share_agent_id, rnn, rnn_c, actions, value_preds, returns, masks,
         active_masks, old_logp, adv_targ, available) = sample
        for p in params:
            p.grad = None
        x, _ = actor.features(obs, node_obs, adj, agent_id, rnn, masks)
        logp = torch.log_softmax(actor.action_out(x).masked_fill(available == 0, -1e10), -1).gather(1, actions.long())
        values, _ = critic(share_obs, node_obs, adj, agent_id, rnn_c, masks)
        ratio = torch.exp(logp - old_logp)
        loss = -(torch.min(ratio * adv_targ, ratio.clamp(0.8, 1.2) * adv_targ) * active_masks).sum() / active_masks.sum()
        loss = loss + (((values - returns) ** 2) * active_masks).sum() / active_masks.sum()
        loss.backward()
        grads = [p.grad for p in params if p.grad is not None]
        assert grads and all(torch.isfinite(g).all() for g in grads) and any(g.abs().sum() > 0 for g in grads)
        n += 1
    assert n == 4
    env.close()
