"""Fused policy kernels (csrc/fm_policy.cu: gnn_kernel<E, RELU> behind fm_gnn_forward, head_kernel<RELU> behind
fm_policy_head) on the GPU, through the C ABI:

* against the frozen outputs of the UNMODIFIED reference GR_Actor / GR_Critic (tests/golden/policy_n3_o3.npz, produced
  by oracle/make_policy_golden.py): gnn features, log-probs, values at 1e-5 * max(|ref|, 1), actions (argmax) exact;
* the graph network against a float64 copy of the dense torch modules (pinned to the reference by tests/test_policy.py)
  at every compiled entity count E, each under ReLU and Tanh, spreading LayerNorm on / off, 0..2 hidden embed layers,
  1, 2, 3 and 8 convs, node / mean / max / add aggregation, node rows of 2, 11, 13 and 17 features, entity types 0..3,
  adjacency shared by the N ego graphs of an env or one per graph, batches that take the persistent loop round more than
  once; a guard that fails when a compiled E has no case; adjacency values on the edge predicate's boundaries
  (``0 < d < max_edge_dist``) for max_edge_dist 1.0, 0.3 and 3.0; a graph gives the same bits alone, in a slice or in
  the full batch;
* the head against a float64 copy of MLPBase / GRU step / output layer: layer_N 0..2, recurrent or not, feature norm on /
  off, ReLU / Tanh, obs_dim 0 (critic), 7, 11, 16, 1, 2, 5 and 8 actions; the mode is the float64 arg-max (exact ties:
  the lower index); a sampled action lies in the float64 inverse-CDF interval of its uniform, and an action of zero
  probability is never drawn, wherever it sits; 2^20 draws through actor.forward(generator=) pass a chi-square test;
* the rollout collector with the fused path == the collector with the dense path (actions exact on a deterministic
  policy), and the sampled loop (deterministic=False, a seeded generator): two eager episodes and a captured one are
  bitwise identical, and every stored log-prob is the float64 policy's at the stored action.
"""
import ast
import copy
import os
from argparse import Namespace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
TOL = 1e-5


def _close(a, b, tol=TOL):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    err = np.abs(a - b) / np.maximum(np.abs(b), 1.0)
    return bool((err <= tol).all()), float(err.max())


def _flat(a):
    return torch.as_tensor(a.reshape((-1,) + a.shape[2:])).cuda()


def _rel_err(x, ref64):
    return float((torch.abs(x.double() - ref64) / torch.clamp(ref64.abs(), min=1.0)).max())


def _assert_bar(e_fused, e_torch, what):
    """A fused result may be off the float64 truth by at most 3 x torch's own fp32 error (floor 1e-5)."""
    assert e_fused <= max(3.0 * e_torch, TOL), (what, e_fused, e_torch)


def _perturb(module, skip=""):
    """Move the weights away from the init, so that every layer matters and the LayerNorms see small variances (fp32
    round-off is amplified): the fused kernels are then held to the float64 truth as tightly as torch's fp32 is."""
    with torch.no_grad():
        for name, p in module.named_parameters():
            if not (skip and name.startswith(skip)):
                p.add_(0.3 * torch.randn_like(p))
    return module


def test_fused_policy_matches_reference_golden():
    from fair_marl_b200.policy import DenseGraphActor, DenseGraphCritic, PolicyConfig, load_reference_state_dict
    from oracle.make_policy_golden import BASE_ARGS
    z = np.load(os.path.join(GOLDEN, "policy_n3_o3.npz"))
    N, O, B, _ = (int(v) for v in z["meta"])
    cfg = PolicyConfig.from_args(Namespace(**{**BASE_ARGS, "num_agents": N, **ast.literal_eval(str(z["overrides"]))}))
    actor, critic = DenseGraphActor(cfg).eval().cuda(), DenseGraphCritic(cfg).eval().cuda()
    load_reference_state_dict(actor, {k[6:]: z[k] for k in z.files if k.startswith("actor/")})
    load_reference_state_dict(critic, {k[7:]: z[k] for k in z.files if k.startswith("critic/")})
    adj_env = torch.as_tensor(z["in_adj_env"]).cuda().contiguous()
    obs, node, aid = _flat(z["in_obs"]), _flat(z["in_node_obs"]), _flat(z["in_agent_id"])
    rnn, masks = _flat(z["in_rnn_states"]), _flat(z["in_masks"])
    assert actor.gnn_base.fused_available(node) is False            # grad mode: the torch path
    with torch.no_grad():
        assert actor.gnn_base.fused_available(node) and critic.gnn_base.fused_available(node)
        act, logp, h = actor(obs, node, None, aid, rnn, masks, deterministic=True, adj_env=(adj_env, N))
        feat = actor.gnn_base(node, None, aid, adj_env=(adj_env, N))
        val, hc = critic(None, node, None, aid, rnn, masks, adj_env=(adj_env, N))
    assert np.array_equal(act.cpu().numpy(), z["out_actions"])
    for name, got in (("gnn_feat", feat), ("action_log_probs", logp), ("rnn_out", h), ("values", val), ("rnn_out_critic", hc)):
        ok, err = _close(got.cpu().numpy(), z["out_" + name])
        assert ok, (name, err)


# ---- graph network: gnn_kernel<E, RELU> --------------------------------------------------------------------------------
_T = dict(embed_use_ReLU=False, gnn_use_ReLU=False)
# (E, node_feat_dim, aggregation, graphs per adjacency, PolicyConfig overrides + "B": adjacency matrices, default 701).
# Every compiled E runs under ReLU and under Tanh.  The lane mapping depends on E: LPT = 32 / E lanes per target
# (E = 5: 6, E = 6: 5, ... E >= 17: 1), SPL sources per lane, and the q|k|v|skip projection takes nodes 9 at a time.
# M = B * rep above 2 368 (2 x 148 SMs x 8 warps) sends warps round the persistent loop more than once.
GNN_CASES = [
    (9, 11, "node", 3, {}), (9, 11, "mean", 3, {}), (9, 13, "node", 3, {}), (9, 13, "mean", 1, {}),
    (17, 11, "max", 7, dict(embed_layer_N=2, gnn_layer_N=1, embed_use_ReLU=False, gnn_use_ReLU=False, use_feature_normalization=False)),
    (11, 11, "add", 3, dict(embed_layer_N=0, gnn_layer_N=0)),
    (7, 11, "node", 2, {}), (19, 11, "mean", 7, {}), (13, 13, "node", 5, {}),
    (5, 11, "node", 2, dict(B=1200)),
    (5, 2, "mean", 1, dict(_T, embed_layer_N=2, gnn_layer_N=7, use_feature_normalization=False)),
    (6, 13, "max", 1, dict(embed_layer_N=0, gnn_layer_N=1)),
    (6, 17, "node", 2, dict(_T, gnn_layer_N=0, B=1300)),
    (7, 11, "add", 3, dict(_T, embed_layer_N=2)),
    (8, 17, "add", 3, dict(use_feature_normalization=False, gnn_layer_N=7)),
    (8, 11, "node", 3, dict(_T, embed_layer_N=0, max_edge_dist=0.3)),
    (9, 13, "node", 3, dict(_T, use_feature_normalization=False)),
    (10, 11, "node", 5, dict(B=523)),                                 # navigation N = 5, O = 0
    (10, 13, "mean", 4, dict(_T, embed_layer_N=2, gnn_layer_N=1)),    # formation N = 4, O = 2
    (11, 2, "max", 1, dict(_T, gnn_layer_N=7, max_edge_dist=3.0)),
    (12, 13, "node", 5, dict(embed_layer_N=2, gnn_layer_N=0, use_feature_normalization=False)),
    (12, 11, "add", 1, dict(_T, gnn_layer_N=1)),
    (13, 17, "max", 1, dict(_T, embed_layer_N=0)),
    (14, 11, "mean", 6, dict(gnn_layer_N=1, max_edge_dist=0.3)),
    (14, 2, "node", 1, dict(_T, use_feature_normalization=False)),
    (15, 13, "add", 1, dict(embed_layer_N=0, gnn_layer_N=7)),
    (15, 11, "node", 5, dict(_T)),
    (17, 13, "node", 7, dict(use_feature_normalization=False, embed_layer_N=2)),
    (19, 17, "add", 1, dict(_T, embed_layer_N=0, gnn_layer_N=7, use_feature_normalization=False)),
]


def _gnn(aggr, seed, **kw):
    import fair_marl_b200 as fm
    from fair_marl_b200.policy import DenseGNNBase
    cfg = fm.PolicyConfig(**kw)
    if aggr != "node":
        cfg.global_aggr_type = aggr
    torch.manual_seed(seed)
    return _perturb(DenseGNNBase(cfg, "node" if aggr == "node" else "global").eval().cuda())


def _float64_copy(module):
    """The same function in float64.  The predicate compares with the fp32 value of max_edge_dist, as the fp32 paths do."""
    ref = copy.deepcopy(module).double()
    ref.cfg.max_edge_dist = float(np.float32(module.cfg.max_edge_dist))
    return ref


@pytest.mark.parametrize("E,NF,aggr,rep,kw", GNN_CASES)
def test_fused_gnn_matches_dense_modules(E, NF, aggr, rep, kw):
    kw = dict(kw)
    B = kw.pop("B", 701)                                              # several CTAs, ragged last one
    gnn = _gnn(aggr, E * 100 + NF, node_feat_dim=NF, **kw)
    M = B * rep
    g = torch.Generator(device="cuda").manual_seed(7)
    pos = torch.rand(B, E, 2, generator=g, device="cuda") * 2 - 1
    adj_env = torch.cdist(pos, pos).float().contiguous()
    adj_env[0, 1, :] = 5.0; adj_env[0, :, 1] = 5.0; adj_env[0, 1, 1] = 0.0     # a node without edges
    adj_env[1] = 5.0                                                             # a graph without edges
    node = torch.randn(M, E, NF, generator=g, device="cuda")
    node[..., -1] = torch.randint(0, 4, (M, E), generator=g, device="cuda").float()   # entity types 0..3 (3: walls)
    aid = torch.randint(0, E, (M, 1), generator=g, device="cuda")
    with torch.no_grad():
        adj_rep = adj_env.repeat_interleave(rep, dim=0)
        ref32 = gnn(node, adj_rep, aid)
        ref64 = _float64_copy(gnn)(node.double(), adj_rep.double(), aid)
        out = gnn(node, None, aid, adj_env=(adj_env, rep))
        out2 = gnn.forward_fused(node, adj_env, rep, aid)             # deterministic: bit-identical on a second launch
    # the fused kernel is held to the float64 truth as tightly as torch's own fp32 evaluation is (x3, floor 1e-5)
    e_fused, e_torch = _rel_err(out, ref64), _rel_err(ref32, ref64)
    assert e_fused <= max(3.0 * e_torch, TOL), (e_fused, e_torch)
    assert torch.equal(out, out2)


def test_gnn_cases_cover_every_compiled_entity_count():
    """A newly compiled E (FM_GNN_CASES in fm_policy.cu) must get a case under each activation."""
    from fair_marl_b200 import _lib
    lib = _lib.load()
    compiled = {E for E in range(1, 65) if lib.fm_gnn_supported(E, 11)}
    assert compiled
    for relu in (True, False):
        have = {c[0] for c in GNN_CASES if c[4].get("gnn_use_ReLU", True) == relu}
        assert compiled <= have, ("ReLU" if relu else "Tanh", sorted(compiled - have))


@pytest.mark.parametrize("E,max_edge_dist", [(9, 1.0), (5, 0.3), (10, 3.0), (17, 0.3)])
def test_fused_gnn_edge_predicate_boundaries(E, max_edge_dist):
    """process_adj keeps an edge iff 0 < d < max_edge_dist (strict both ways, fp32).  Each graph has one pair (r -> t) at
    a boundary value; the output is the gathered node t, and moving that one pair across the predicate is checked to
    change the float64 output by far more than the tolerance, so a kernel that decides the pair differently fails."""
    gnn = _gnn("node", E, max_edge_dist=max_edge_dist)
    m32 = np.float32(max_edge_dist)
    below = np.nextafter(m32, np.float32(0))
    tiny = np.finfo(np.float32).smallest_subnormal
    # boundary value, and its counterpart on the other side of the predicate at (almost) the same distance
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
    adj[b] = 2 * m32 + 1; adj[b, range(E), range(E)] = 0.0                              # no edges
    adj[b + 1] = rng.uniform(0.05, 0.95, (E, E)) * m32; adj[b + 1, range(E), range(E)] = 0.0   # complete graph
    flip[b:] = adj[b:]
    assert np.signbit(adj[3 * len(pairs), pairs[0][0], pairs[0][1]])                     # -0.0 survived
    g = torch.Generator(device="cuda").manual_seed(E)
    node = torch.randn(B, E, 11, generator=g, device="cuda")
    node[..., -1] = torch.randint(0, 4, (B, E), generator=g, device="cuda").float()
    adj_t, flip_t, aid_t = (torch.from_numpy(x).cuda() for x in (adj, flip, aid))
    with torch.no_grad():
        ref = _float64_copy(gnn)
        ref64, ref64_flip = ref(node.double(), adj_t.double(), aid_t), ref(node.double(), flip_t.double(), aid_t)
        ref32 = gnn(node, adj_t, aid_t)
        out = gnn.forward_fused(node.contiguous(), adj_t.contiguous(), 1, aid_t)
    moved = (torch.abs(ref64_flip - ref64) / torch.clamp(ref64.abs(), min=1.0)).amax(dim=1)[:b]
    assert (moved > 100 * TOL).all(), float(moved.min())
    _assert_bar(_rel_err(out, ref64), _rel_err(ref32, ref64), "gnn features")


@pytest.mark.parametrize("E,rep,aggr", [(5, 2, "node"), (10, 1, "mean"), (17, 3, "node")])
def test_fused_gnn_is_batch_invariant(E, rep, aggr):
    """A graph's output does not depend on where it sits in the launch: alone, in a slice starting at an (unaligned)
    offset, in the first or a later round of the persistent loop of the full batch -- the same bits."""
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
        full = gnn.forward_fused(node, adj, rep, aid)
        assert torch.equal(full, gnn.forward_fused(node, adj, rep, aid))
        for m in (0, 1, 2367, 2368, M - 1):
            k = m // rep
            alone = gnn.forward_fused(node[m:m + 1], adj[k:k + 1], 1, aid[m:m + 1] if aid is not None else None)
            assert torch.equal(alone[0], full[m]), m
        k0 = 37
        part = gnn.forward_fused(node[k0 * rep:], adj[k0:], rep, aid[k0 * rep:] if aid is not None else None)
        assert torch.equal(part, full[k0 * rep:])


# ---- head: head_kernel<RELU> ---------------------------------------------------------------------------------------------
# (actor / critic, layer_N, recurrent, feature norm, ReLU, obs_dim, actions, rows).  16 warps per CTA, one CTA per SM:
# more than 148 x 16 = 2 368 rows take the persistent loop round again.
HEAD_CASES = [
    ("actor", 1, True, True, True, 7, 5, 701),
    ("actor", 0, False, True, False, 11, 8, 2500),
    ("actor", 2, True, False, True, 16, 2, 333),
    ("actor", 2, True, True, False, 7, 1, 129),
    ("actor", 1, False, False, True, 11, 5, 64),
    ("actor", 2, False, False, False, 16, 8, 2777),
    ("critic", 2, False, True, False, 0, 1, 1000),
    ("critic", 0, True, False, True, 0, 1, 517),
]


def _head_net(kind, layer_N, recurrent, feat_norm, relu, obs_dim, A, seed):
    import fair_marl_b200 as fm
    cfg = fm.PolicyConfig(obs_dim=obs_dim, action_dim=A, layer_N=layer_N, use_recurrent_policy=recurrent,
                          use_feature_normalization=feat_norm, use_ReLU=relu)
    torch.manual_seed(seed)
    net = _perturb((fm.DenseGraphActor if kind == "actor" else fm.DenseGraphCritic)(cfg).eval().cuda(), skip="gnn_base.")
    assert net.head_supported()
    return net


def _head_inputs(net, M, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    obs_dim = net._head_in - 16
    obs = 2 * torch.randn(M, obs_dim, generator=g, device="cuda") if obs_dim else None
    nbd = 2 * torch.randn(M, 16, generator=g, device="cuda")
    rnn = torch.randn(M, 1, 64, generator=g, device="cuda")
    masks = (torch.rand(M, 1, generator=g, device="cuda") < 0.7).float()          # mixed 0 / 1
    assert 0 < masks.sum() < M
    return obs, nbd, rnn, masks


def _head_reference(net, obs, nbd, rnn, masks):
    """MLPBase -> GRU step -> output layer of `net` on the inputs of `_run_head`: (outputs, pre-LayerNorm hidden state)."""
    x = nbd if obs is None else torch.cat([obs, nbd], dim=1)
    x, h = net.base(x), None
    if net.recurrent:
        x, h = net.rnn(x, rnn, masks)
    return net._out_linear()(x), h


def _f64(*xs):
    return [None if x is None else x.double() for x in xs]


def _boundary_uniforms(C, seed):
    """One u per row (fp32): 0, 1 - 2^-24, the fp32 neighbours just below and just above a float64 CDF boundary, or a
    uniform draw.  C [M, A] float64 CDF."""
    M, A = C.shape
    rng = np.random.default_rng(seed)
    Cn = C.cpu().numpy()
    top = np.float32(1.0 - 2.0 ** -24)
    u = rng.random(M).astype(np.float32)
    for m in range(M):
        kind, b = m % 6, Cn[m, (m // 6) % A]
        if kind == 0:
            u[m] = 0.0
        elif kind == 1:
            u[m] = top
        elif kind in (2, 3):
            b32 = np.float32(b)
            if kind == 2:
                u[m] = b32 if b32 < b else np.nextafter(b32, np.float32(0))
            else:
                u[m] = min(b32 if b32 > b else np.nextafter(b32, np.float32(2)), top)
    return torch.from_numpy(u).cuda()


def _check_sampled(act, u, logits64, slack=1e-5):
    """The inverse-CDF contract: C[a-1] - slack <= u < C[a] + slack for the float64 CDF C, and no action of float64
    probability below 1e-30."""
    p = torch.softmax(logits64, dim=1)
    C = torch.cumsum(p, dim=1)
    a = act.view(-1, 1)
    lo = torch.where(a > 0, C.gather(1, (a - 1).clamp(min=0)), torch.zeros_like(C[:, :1]))[:, 0]
    hi = C.gather(1, a)[:, 0]
    ud = u.double()
    bad = ~((lo - slack <= ud) & (ud < hi + slack))
    assert not bad.any(), [(int(m), float(u[m]), int(act[m]), C[m].tolist()) for m in bad.nonzero()[:5, 0]]
    pa = p.gather(1, a)[:, 0]
    assert (pa >= 1e-30).all(), [(int(m), float(u[m]), int(act[m]), p[m].tolist()) for m in (pa < 1e-30).nonzero()[:5, 0]]


@pytest.mark.parametrize("kind,layer_N,recurrent,feat_norm,relu,obs_dim,A,M", HEAD_CASES)
def test_fused_head_matches_float64(kind, layer_N, recurrent, feat_norm, relu, obs_dim, A, M):
    net = _head_net(kind, layer_N, recurrent, feat_norm, relu, obs_dim, A, seed=M)
    critic = kind == "critic"
    if A >= 5:                                           # output row A-1 = row 1: exactly tied logits on every row
        with torch.no_grad():
            net.action_out.weight[A - 1] = net.action_out.weight[1]
            net.action_out.bias[A - 1] = net.action_out.bias[1]
    obs, nbd, rnn, masks = _head_inputs(net, M, seed=A)
    with torch.no_grad():
        out32, h32 = _head_reference(net, obs, nbd, rnn, masks)
        out64, h64 = _head_reference(copy.deepcopy(net).double(), *_f64(obs, nbd, rnn, masks))
        res = net._run_head(obs, nbd, rnn, masks, None, critic=critic)
    bar = lambda got, r32, r64, what: _assert_bar(_rel_err(got, r64), _rel_err(r32, r64), what)
    if recurrent:
        bar(res[-1], h32, h64, "rnn_out")
    else:
        assert res[-1] is rnn                                          # passed through
    if critic:
        bar(res[0], out32, out64, "values")
        return
    lp32, lp64 = torch.log_softmax(out32, dim=1), torch.log_softmax(out64, dim=1)
    # deterministic: FixedCategorical.mode, the first maximum
    act, logp = res[0][:, 0], res[1]
    bar(logp, lp32.gather(1, res[0]), lp64.gather(1, res[0]), "logp (mode)")
    L = out64[:, :A - 1] if A >= 5 else out64                           # the duplicate column never wins a tie
    top = L.max(dim=1).values
    near = L >= (top - 1e-4 * top.abs().clamp(min=1.0)).unsqueeze(1)
    clear = near.sum(dim=1) == 1
    assert torch.equal(act[clear], L.argmax(dim=1)[clear]), int((act[clear] != L.argmax(dim=1)[clear]).sum())
    assert near.gather(1, act.clamp(max=L.shape[1] - 1).view(-1, 1)).all()
    if A >= 5:
        assert (act != A - 1).all() and (act == 1).any()                # ties: the lower index, as torch's argmax
    # sampled: inverse CDF of the caller's uniforms
    u = _boundary_uniforms(torch.cumsum(torch.softmax(out64, dim=1), dim=1), seed=M)
    with torch.no_grad():
        act_s, logp_s, _ = net._run_head(obs, nbd, rnn, masks, u, critic=False)
    _check_sampled(act_s[:, 0], u, out64)
    bar(logp_s, lp32.gather(1, act_s), lp64.gather(1, act_s), "logp (sampled)")
    if A > 1:
        assert len(torch.unique(act_s)) > 1


@pytest.mark.parametrize("where", ["first", "middle", "last"])
def test_head_sampler_never_draws_a_zero_probability_action(where):
    """An action whose logit sits 200 below the rest has probability ~1e-87: torch.multinomial never draws it, and
    neither may the kernel -- in particular not when u = 1 - 2^-24 lies above the fp32 sum of the probabilities."""
    A, M = 5, 20000
    z = {"first": 0, "middle": 2, "last": A - 1}[where]
    net = _head_net("actor", 1, True, True, True, 7, A, seed=5)
    with torch.no_grad():
        net.action_out.weight[z] = 0.0
        net.action_out.bias[z] = -200.0
    obs, nbd, rnn, masks = _head_inputs(net, M, seed=11)
    u = torch.rand(M, generator=torch.Generator(device="cuda").manual_seed(3), device="cuda")
    u[: M // 3] = 0.0
    u[M // 3: 2 * M // 3] = 1.0 - 2.0 ** -24
    with torch.no_grad():
        out64, _ = _head_reference(copy.deepcopy(net).double(), *_f64(obs, nbd, rnn, masks))
        act, logp, _ = net._run_head(obs, nbd, rnn, masks, u, critic=False)
    assert (torch.softmax(out64, dim=1)[:, z] < 1e-30).all()
    drawn = int((act[:, 0] == z).sum())
    assert drawn == 0, f"the zero-probability action {z} was drawn on {drawn} of {M} rows (log-prob {float(logp.min()):.1f})"
    _check_sampled(act[:, 0], u, out64)


def test_fused_actor_sampling_matches_float64_distribution():
    """2^20 draws of one row through actor.forward(deterministic=False, generator=...) on the fused path: a chi-square test
    against the float64 probabilities of that row (fixed seed, so the outcome is fixed)."""
    from scipy.stats import chi2
    import fair_marl_b200 as fm
    E, N, B = 9, 3, 64
    torch.manual_seed(21)
    actor = _perturb(fm.DenseGraphActor(fm.PolicyConfig(num_agents=N)).eval().cuda())
    with torch.no_grad():
        actor.action_out.weight.mul_(0.3)                                # a spread-out distribution
    g = torch.Generator(device="cuda").manual_seed(17)
    pos = torch.rand(B, E, 2, generator=g, device="cuda") * 2 - 1
    adj = torch.cdist(pos, pos).float()
    node = torch.randn(B * N, E, 11, generator=g, device="cuda")
    node[..., -1] = torch.randint(0, 4, (B * N, E), generator=g, device="cuda").float()
    obs = torch.randn(B * N, 7, generator=g, device="cuda")
    aid = torch.arange(N, device="cuda").repeat(B).view(-1, 1)
    rnn = torch.randn(B * N, 1, 64, generator=g, device="cuda")
    masks = torch.ones(B * N, 1, device="cuda")
    with torch.no_grad():
        ref = copy.deepcopy(actor).double()
        x, _ = ref.features(obs.double(), node.double(), adj.repeat_interleave(N, 0).double(), aid, rnn.double(), masks.double())
        p = torch.softmax(ref.action_out(x), dim=1)
    m = int(p.min(dim=1).values.argmax())                               # the row whose rarest action is most likely
    p = p[m]
    assert float(p.min()) > 0.01
    n = 1 << 20
    rows = lambda t: t[m:m + 1].expand(n, *t.shape[1:]).contiguous()
    with torch.no_grad():
        act, logp, _ = actor(rows(obs), rows(node), None, rows(aid), rows(rnn), rows(masks), deterministic=False,
                             generator=torch.Generator(device="cuda").manual_seed(2024), adj_env=(adj[m // N:m // N + 1].contiguous(), n))
    counts = torch.bincount(act[:, 0], minlength=5).double()
    expected = n * p
    stat = float(((counts - expected) ** 2 / expected).sum())
    pval = float(chi2.sf(stat, df=4))
    assert pval > 1e-3, (stat, pval, counts.tolist(), expected.tolist())
    assert torch.allclose(logp[:, 0].double(), torch.log(p)[act[:, 0]], rtol=0, atol=1e-4)


# ---- rollout collector ----------------------------------------------------------------------------------------------------
def test_collector_fused_equals_dense():
    import fair_marl_b200 as fm
    from oracle.navgraph import NavConfig
    from parity_util import sim_config_from
    cfg = NavConfig(num_agents=3, num_obstacles=3, episode_length=8)
    outs = []
    for fused in (True, False):
        env = fm.B200GraphVecEnv(sim_config_from(cfg), num_envs=160, seed=11)
        pc = fm.PolicyConfig(num_agents=3)
        torch.manual_seed(0)
        actor, critic = fm.DenseGraphActor(pc).to(env.device).eval(), fm.DenseGraphCritic(pc).to(env.device).eval()
        with torch.no_grad():
            actor.action_out.weight.mul_(100.0)
        col = fm.RolloutCollector(env, actor, critic, deterministic=True, fused=fused)
        assert col.fused is fused
        col.warmup(); col.run()
        torch.cuda.synchronize()
        outs.append((col.buffer.actions_env.clone(), col.buffer.value_preds.clone(), col.buffer.obs.clone()))
        env.close()
    assert torch.equal(outs[0][0], outs[1][0])                        # same actions => same trajectories
    assert torch.equal(outs[0][2], outs[1][2])
    ok, err = _close(outs[0][1].cpu().numpy(), outs[1][1].cpu().numpy(), 2e-5)
    assert ok, err


def _sampled_collector(family, use_graph):
    """Navigation N = 3 / O = 3 (E = 9) or formation N = 5 / O = 2 (E = 12); sampled actions from a seeded generator."""
    import fair_marl_b200 as fm
    if family == "navigation":
        from oracle.navgraph import NavConfig
        from parity_util import sim_config_from
        env = fm.B200GraphVecEnv(sim_config_from(NavConfig(num_agents=3, num_obstacles=3, episode_length=10)), num_envs=128, seed=11)
        pc = fm.PolicyConfig(num_agents=3)
    else:
        cfg = fm.FormationSimConfig(num_agents=5, num_obstacles=2, goal_rew=30.0, collision_rew=30.0, episode_length=10)
        env = fm.B200FormationVecEnv(cfg, num_envs=128, seed=11)
        pc = fm.PolicyConfig(num_agents=5, obs_dim=11, node_feat_dim=13)
    torch.manual_seed(0)
    actor, critic = fm.DenseGraphActor(pc).to(env.device).eval(), fm.DenseGraphCritic(pc).to(env.device).eval()
    with torch.no_grad():
        actor.action_out.weight.mul_(30.0)                               # a confident policy: many near-zero probabilities
    col = fm.RolloutCollector(env, actor, critic, deterministic=False,
                              generator=torch.Generator(device=env.device).manual_seed(99))
    assert col.fused
    col.warmup(); col.run(); col.buffer.after_update()
    if use_graph:
        col.capture()
    col.run(); col.buffer.after_update(); col.run()                     # the last two episodes replay the graph
    torch.cuda.synchronize()
    b = col.buffer
    fields = [x.clone() for x in (b.obs, b.node_obs, b.adj_env, b.rewards, b.dones, b.actions_env, b.rnn_states, b.masks,
                                  b.value_preds, b.action_log_probs)]
    return env, actor, b, fields


@pytest.mark.parametrize("family", ["navigation", "formation"])
def test_sampled_collector_is_reproducible_and_follows_the_float64_policy(family):
    env, actor, b, eager = _sampled_collector(family, use_graph=False)
    env2, _, _, eager2 = _sampled_collector(family, use_graph=False)
    env3, _, _, graph = _sampled_collector(family, use_graph=True)
    for x, y, z in zip(eager, eager2, graph):
        assert torch.equal(x, y)                                         # same seed, same bits
        assert torch.equal(x, z)                                         # the captured generator state replays the draws
    # every stored (slab, action): the float64 dense policy on the buffer's own inputs
    T, B, N, E = b.episode_length, b.n_rollout_threads, b.num_agents, b.num_entities
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
    assert (lp64 > np.log(1e-30)).all(), float(lp64.min())              # no action of float64 probability below 1e-30
    _assert_bar(_rel_err(stored, lp64), _rel_err(lp32, lp64), "stored action_log_probs")
    assert (lp64 < -0.1).any()                                           # draws other than the mode
    for e in (env, env2, env3):
        e.close()
