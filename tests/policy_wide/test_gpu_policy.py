"""The CTA-per-graph mapping of the fused graph network (csrc/fm_policy.cu: gnn_wide_kernel<EMAX, RELU>, selected by
FmGnnConfig.mapping = 2, and by mapping 0 wherever the warp-per-graph kernel is not compiled), on the GPU:

* every E from 2 to 64 under ReLU and under Tanh against a float64 copy of the dense modules, with the bar of
  tests/test_gpu_policy.py (at most 3 x torch's own fp32 error, floor 1e-5).  The cases spread LayerNorm on / off,
  0..2 hidden embed layers, 1, 2, 3 and 8 convs (8 at E = 64), node / mean / max / add aggregation, node rows of 2, 11,
  13 and 17 features, entity types 0..3, one adjacency per graph or per N graphs, a node without edges, a graph without
  edges, a complete graph, and batches that take the persistent loop round more than once;
* a guard: fm_gnn_mapping covers exactly 2 <= E <= 64, and every such E has a case under each activation;
* auto selection: mapping 0 gives the bits of mapping 1 where the warp kernel is compiled, else those of mapping 2;
* the edge predicate 0 < d < max_edge_dist on its boundary values at E = 35 and 64;
* batch invariance and a second launch: identical bits;
* the rollout collector at navigation N = 16 / O = 3 (E = 35) and formation N = 7 / O = 8 / W = 2 (E = 24): fused by
  default and equal to the dense path, and the sampled loop at E = 35 reproducible, captured or eager, and following the
  float64 policy.
"""
import copy

import numpy as np
import pytest
import torch

from test_gpu_policy import TOL, _assert_bar, _close, _float64_copy, _gnn, _rel_err

pytestmark = pytest.mark.gpu

_T = dict(embed_use_ReLU=False, gnn_use_ReLU=False)
_NF = (2, 11, 13, 17)
_AGGR = ("node", "mean", "max", "add")
_CONVS = (0, 1, 2, 7)                                   # gnn_layer_N: 1, 2, 3 and 8 convs


def _wide_cases():
    """(E, node_feat_dim, aggregation, graphs per adjacency, PolicyConfig overrides + "B": adjacency matrices) for every E
    in 2..64, once under ReLU and once under Tanh.  The knobs cycle with different periods so that they meet in many
    combinations; EMAX = 32 serves E <= 32 with 4 threads per target, EMAX = 64 the rest with 2."""
    cases = []
    for E in range(2, 65):
        for relu in (True, False):
            k = 2 * E + (0 if relu else 1)
            kw = {} if relu else dict(_T)
            kw.update(embed_layer_N=k % 3, gnn_layer_N=_CONVS[(k // 3) % 4])
            if E == 64 and not relu:
                # the largest blob (92.5 KB) beside the largest scratch.  Under Tanh: with ReLU and nothing bounding the
                # activations between 8 convs, torch's own fp32 result at E = 64 is 8-9 % off float64, so there is no fp32
                # value to hold a kernel to
                kw["gnn_layer_N"] = 7
            if (k // 2) % 2:
                kw["use_feature_normalization"] = False
            if k % 7 == 3:
                kw["max_edge_dist"] = 0.3
            elif k % 7 == 5:
                kw["max_edge_dist"] = 3.0
            rep = 1 if k % 2 == 0 else max(2, (E - 3) // 2)          # one adjacency per graph, or per N ego graphs
            kw["B"] = 1100 // rep + 3 if k % 5 == 0 else max(8, 160 // rep)
            cases.append((E, _NF[k % 4], _AGGR[(k // 4) % 4], rep, kw))
    return cases


WIDE_CASES = _wide_cases()


def _inputs(B, rep, E, NF, seed):
    M = B * rep
    g = torch.Generator(device="cuda").manual_seed(seed)
    pos = torch.rand(B, E, 2, generator=g, device="cuda") * 2 - 1
    adj_env = torch.cdist(pos, pos).float().contiguous()
    adj_env[0, 1, :] = 5.0; adj_env[0, :, 1] = 5.0; adj_env[0, 1, 1] = 0.0     # a node without edges
    adj_env[1] = 5.0                                                             # a graph without edges
    full = torch.rand(E, E, generator=g, device="cuda") * 0.2 + 0.05             # a complete graph (d < 0.3 everywhere)
    adj_env[2] = torch.minimum(full, full.t()).fill_diagonal_(0.0)
    node = torch.randn(M, E, NF, generator=g, device="cuda")
    node[..., -1] = torch.randint(0, 4, (M, E), generator=g, device="cuda").float()   # entity types 0..3 (3: walls)
    aid = torch.randint(0, E, (M, 1), generator=g, device="cuda")
    return adj_env, node, aid


RELABELLINGS = 7


def _errors_over_labellings(gnn, node, adj_env, rep, aid, ref64, seed, fused_aid=True):
    """(kernel error, torch fp32 error) on these graphs, each the largest over the given node labelling and RELABELLINGS
    others.  Relabelling the nodes (one permutation of node rows, adjacency rows and columns, and the gathered index)
    leaves the function unchanged but reorders every fp32 sum over nodes.  Without LayerNorm, or with LayerNorms that see
    small variances, and E in the 30s to 60s, one fp32 evaluation is a draw from a wide distribution: at E = 37 with two
    hidden embed layers torch's own error ranges from 1.5e-5 to 8.3e-5 over eight labellings of the same graphs, and the
    kernel's from 1.6e-5 to 7.1e-5; with 8 convs and no normalization between them (E = 53) both range over a factor of
    seven.  Both implementations are therefore compared over the same eight labellings."""
    E = node.shape[1]
    g = torch.Generator().manual_seed(seed)
    e_fused, e_torch = [], []
    for k in range(1 + RELABELLINGS):
        perm = (torch.arange(E) if k == 0 else torch.randperm(E, generator=g)).to(node.device)
        inv = torch.argsort(perm)
        n2, a2, i2 = node[:, perm].contiguous(), adj_env[:, perm][:, :, perm].contiguous(), inv[aid]
        e_torch.append(_rel_err(gnn(n2, a2.repeat_interleave(rep, dim=0), i2), ref64))
        e_fused.append(_rel_err(gnn.forward_fused(n2, a2, rep, i2 if fused_aid else None, mapping=2), ref64))
    return max(e_fused), max(e_torch)


@pytest.mark.parametrize("E,NF,aggr,rep,kw", WIDE_CASES)
def test_wide_gnn_matches_dense_modules(E, NF, aggr, rep, kw):
    kw = dict(kw)
    B = kw.pop("B")
    gnn = _gnn(aggr, E * 100 + NF, node_feat_dim=NF, **kw)
    adj_env, node, aid = _inputs(B, rep, E, NF, seed=E)
    with torch.no_grad():
        adj_rep = adj_env.repeat_interleave(rep, dim=0)
        ref64 = _float64_copy(gnn)(node.double(), adj_rep.double(), aid)
        e_fused, e_torch = _errors_over_labellings(gnn, node, adj_env, rep, aid, ref64, seed=E, fused_aid=aggr == "node")
        out = gnn.forward_fused(node, adj_env, rep, aid if aggr == "node" else None, mapping=2)
        out2 = gnn.forward_fused(node, adj_env, rep, aid if aggr == "node" else None, mapping=2)
    assert e_fused <= max(3.0 * e_torch, TOL), (e_fused, e_torch)
    assert torch.equal(out, out2)


def test_wide_cases_cover_every_served_entity_count():
    """fm_gnn_mapping is nonzero exactly for 2 <= E <= 64, and every such E has a case under each activation."""
    from fair_marl_b200 import _lib
    lib = _lib.load()
    served = {E for E in range(0, 80) if lib.fm_gnn_mapping(E, 11)}
    assert served == set(range(2, 65))
    assert lib.fm_gnn_mapping(1, 11) == 0 and lib.fm_gnn_mapping(65, 11) == 0
    for relu in (True, False):
        have = {c[0] for c in WIDE_CASES if c[4].get("gnn_use_ReLU", True) == relu}
        assert served <= have, ("ReLU" if relu else "Tanh", sorted(served - have))
    assert any(c[0] == 64 and c[4].get("gnn_layer_N") == 7 for c in WIDE_CASES)


def test_auto_mapping_selects_warp_kernel_where_compiled_else_wide():
    """mapping 0 == mapping 1 bit for bit where the warp kernel is compiled (existing results do not change), and == mapping 2
    everywhere else; mapping 1 is refused where the warp kernel is not compiled."""
    from fair_marl_b200 import _lib
    lib = _lib.load()
    for E in range(2, 65):
        gnn = _gnn("node", E, node_feat_dim=11)
        adj_env, node, aid = _inputs(300, 2, E, 11, seed=E + 1000)
        with torch.no_grad():
            auto = gnn.forward_fused(node, adj_env, 2, aid)
            wide = gnn.forward_fused(node, adj_env, 2, aid, mapping=2)
            if lib.fm_gnn_supported(E, 11):
                assert lib.fm_gnn_mapping(E, 11) == 1
                assert torch.equal(auto, gnn.forward_fused(node, adj_env, 2, aid, mapping=1)), E
            else:
                assert lib.fm_gnn_mapping(E, 11) == 2
                assert torch.equal(auto, wide), E
                with pytest.raises(_lib.FairMarlError, match="mapping 1"):
                    gnn.forward_fused(node, adj_env, 2, aid, mapping=1)


@pytest.mark.parametrize("E,max_edge_dist", [(35, 1.0), (35, 0.3), (64, 1.0), (64, 3.0)])
def test_wide_gnn_edge_predicate_boundaries(E, max_edge_dist):
    """As test_fused_gnn_edge_predicate_boundaries, on the CTA-per-graph kernel: one pair (r -> t) per graph at fp32
    max_edge_dist, its predecessor, 0, -0 or the smallest denormal; flipping that pair across the predicate moves the
    float64 output far beyond the tolerance."""
    gnn = _gnn("node", E, max_edge_dist=max_edge_dist)
    m32 = np.float32(max_edge_dist)
    below = np.nextafter(m32, np.float32(0))
    tiny = np.finfo(np.float32).smallest_subnormal
    values = [(m32, below), (below, m32), (np.float32(0.0), tiny), (np.float32(-0.0), tiny), (tiny, np.float32(0.0))]
    pairs = [(r, t) for t in range(E) for r in {(t + 1) % E, (t + E // 2) % E, (t + E - 1) % E} - {t}]
    rng = np.random.default_rng(E)
    B = len(values) * len(pairs) + 2
    adj = np.where(rng.random((B, E, E)) < 0.4, rng.uniform(0.05, 0.95, (B, E, E)) * m32, 2 * m32 + 1).astype(np.float32)
    adj = np.minimum(adj, adj.transpose(0, 2, 1))
    adj[:, range(E), range(E)] = 0.0
    flip = adj.copy()
    aid = np.zeros((B, 1), np.int64)
    b = 0
    for v, other in values:
        for r, t in pairs:
            adj[b, r, t], flip[b, r, t], aid[b] = v, other, t
            b += 1
    adj[b] = 2 * m32 + 1; adj[b, range(E), range(E)] = 0.0
    adj[b + 1] = rng.uniform(0.05, 0.95, (E, E)) * m32; adj[b + 1, range(E), range(E)] = 0.0
    flip[b:] = adj[b:]
    assert np.signbit(adj[3 * len(pairs), pairs[0][0], pairs[0][1]])
    g = torch.Generator(device="cuda").manual_seed(E)
    node = torch.randn(B, E, 11, generator=g, device="cuda")
    node[..., -1] = torch.randint(0, 4, (B, E), generator=g, device="cuda").float()
    adj_t, flip_t, aid_t = (torch.from_numpy(x).cuda() for x in (adj, flip, aid))
    with torch.no_grad():
        ref = _float64_copy(gnn)
        ref64, ref64_flip = ref(node.double(), adj_t.double(), aid_t), ref(node.double(), flip_t.double(), aid_t)
        e_fused, e_torch = _errors_over_labellings(gnn, node.contiguous(), adj_t.contiguous(), 1, aid_t, ref64, seed=E)
    moved = (torch.abs(ref64_flip - ref64) / torch.clamp(ref64.abs(), min=1.0)).amax(dim=1)[:b]
    assert (moved > 100 * TOL).all(), float(moved.min())
    _assert_bar(e_fused, e_torch, "gnn features")


@pytest.mark.parametrize("E,rep,aggr", [(35, 16, "node"), (64, 1, "mean"), (24, 7, "node"), (3, 1, "max")])
def test_wide_gnn_is_batch_invariant(E, rep, aggr):
    """A graph gives the same bits alone, in a slice at an unaligned offset, and in the full batch, whose CTAs take the
    persistent loop round several times (grid <= 2 CTAs x 148 SMs); a second launch gives the same bits."""
    gnn = _gnn(aggr, 3 * E, node_feat_dim=13)
    B = 2400 // rep + 7
    M = B * rep
    g = torch.Generator(device="cuda").manual_seed(E)
    pos = torch.rand(B, E, 2, generator=g, device="cuda") * 2 - 1
    adj = torch.cdist(pos, pos).float().contiguous()
    node = torch.randn(M, E, 13, generator=g, device="cuda")
    node[..., -1] = torch.randint(0, 4, (M, E), generator=g, device="cuda").float()
    aid = torch.randint(0, E, (M, 1), generator=g, device="cuda") if aggr == "node" else None
    with torch.no_grad():
        full = gnn.forward_fused(node, adj, rep, aid, mapping=2)
        assert torch.equal(full, gnn.forward_fused(node, adj, rep, aid, mapping=2))
        for m in (0, 1, 295, 296, 297, 1500, M - 1):
            k = m // rep
            alone = gnn.forward_fused(node[m:m + 1], adj[k:k + 1], 1, aid[m:m + 1] if aid is not None else None, mapping=2)
            assert torch.equal(alone[0], full[m]), m
        k0 = 37
        part = gnn.forward_fused(node[k0 * rep:], adj[k0:], rep, aid[k0 * rep:] if aid is not None else None, mapping=2)
        assert torch.equal(part, full[k0 * rep:])


# ---- rollout collector at shapes only the CTA-per-graph kernel serves --------------------------------------------------
def _env_policy(family, num_envs, seed=11, episode_length=8, scale=100.0):
    import fair_marl_b200 as fm
    if family == "navigation":                                            # BASELINE C4: N = 16, O = 3 -> E = 35
        from oracle.navgraph import NavConfig
        from parity_util import sim_config_from
        env = fm.B200GraphVecEnv(sim_config_from(NavConfig(num_agents=16, num_obstacles=3, episode_length=episode_length)),
                                 num_envs=num_envs, seed=seed)
        pc = fm.PolicyConfig(num_agents=16)
    else:                                                                 # formation N = 7, O = 8, W = 2 -> E = 24
        cfg = fm.FormationSimConfig(num_agents=7, num_obstacles=8, num_walls=2, goal_rew=30.0, collision_rew=30.0,
                                    episode_length=episode_length)
        env = fm.B200FormationVecEnv(cfg, num_envs=num_envs, seed=seed)
        pc = fm.PolicyConfig(num_agents=7, obs_dim=11, node_feat_dim=13)
    torch.manual_seed(0)
    actor, critic = fm.DenseGraphActor(pc).to(env.device).eval(), fm.DenseGraphCritic(pc).to(env.device).eval()
    with torch.no_grad():
        actor.action_out.weight.mul_(scale)
    return fm, env, actor, critic


@pytest.mark.parametrize("family,E", [("navigation", 35), ("formation", 24)])
def test_collector_fused_equals_dense_at_wide_shapes(family, E):
    from fair_marl_b200 import _lib
    assert _lib.load().fm_gnn_mapping(E, 13 if family == "formation" else 11) == 2
    outs = []
    for fused in (None, False):
        fm, env, actor, critic = _env_policy(family, 96)
        col = fm.RolloutCollector(env, actor, critic, deterministic=True, fused=fused)
        assert col.buffer.num_entities == E
        assert col.fused is (fused is None)                               # fused by default at this shape
        col.warmup(); col.run()
        torch.cuda.synchronize()
        outs.append((col.buffer.actions_env.clone(), col.buffer.value_preds.clone(), col.buffer.obs.clone()))
        env.close()
    assert torch.equal(outs[0][0], outs[1][0])                            # same actions => same trajectories
    assert torch.equal(outs[0][2], outs[1][2])
    ok, err = _close(outs[0][1].cpu().numpy(), outs[1][1].cpu().numpy(), 2e-5)
    assert ok, err


def _sampled_run(use_graph):
    fm, env, actor, critic = _env_policy("navigation", 48, episode_length=10, scale=30.0)
    col = fm.RolloutCollector(env, actor, critic, deterministic=False,
                              generator=torch.Generator(device=env.device).manual_seed(99))
    assert col.fused
    col.warmup(); col.run(); col.buffer.after_update()
    if use_graph:
        col.capture()
    col.run(); col.buffer.after_update(); col.run()
    torch.cuda.synchronize()
    b = col.buffer
    fields = [x.clone() for x in (b.obs, b.node_obs, b.adj_env, b.rewards, b.dones, b.actions_env, b.rnn_states, b.masks,
                                  b.value_preds, b.action_log_probs)]
    return env, actor, b, fields


def test_sampled_collector_at_e35_is_reproducible_and_follows_the_float64_policy():
    env, actor, b, eager = _sampled_run(False)
    env2, _, _, eager2 = _sampled_run(False)
    env3, _, _, graph = _sampled_run(True)
    for x, y, z in zip(eager, eager2, graph):
        assert torch.equal(x, y)
        assert torch.equal(x, z)
    T, B, N, E = b.episode_length, b.n_rollout_threads, b.num_agents, b.num_entities
    assert E == 35
    M = B * N
    ref = copy.deepcopy(actor).double()
    lp64, lp32 = [], []
    with torch.no_grad():
        for t in range(T):
            args = (b.obs[t].view(M, -1), b.node_obs[t].view(M, E, -1), b.adj_env[t].repeat_interleave(N, 0),
                    b.agent_id[t].reshape(M, 1), b.rnn_states[t].view(M, 1, -1), b.masks[t].view(M, 1))
            a = b.actions_env[t].view(M, 1).long()
            x, _ = ref.features(*[v.double() if v.is_floating_point() else v for v in args])
            lp64.append(torch.log_softmax(ref.action_out(x), dim=1).gather(1, a))
            x, _ = actor.features(*args)
            lp32.append(torch.log_softmax(actor.action_out(x), dim=1).gather(1, a))
    lp64, lp32 = torch.cat(lp64), torch.cat(lp32)
    stored = b.action_log_probs[:T].reshape(-1, 1)
    assert (lp64 > np.log(1e-30)).all(), float(lp64.min())
    _assert_bar(_rel_err(stored, lp64), _rel_err(lp32, lp64), "stored action_log_probs")
    assert (lp64 < -0.1).any()
    for e in (env, env2, env3):
        e.close()
