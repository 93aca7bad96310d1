"""The centralised-observation (use_cent_obs) and per-agent (critic_graph_aggr='node') critics on the GPU:

* the wide critic head (csrc/fm_policy.cu critic_head_kernel behind fm_critic_head) against a float64 copy of MLPBase +
  GRU step + v_out, with the bar of tests/test_gpu_policy.py (at most 3 x torch's own fp32 error, floor 1e-5), at every
  (family, N, configuration) the fused critic serves: navigation N = 2..32 and formation N = 2..7, each with cent_obs +
  global pool, node gather, and cent_obs + node gather; the cases spread layer_N 0..2, recurrent or not, feature norm on /
  off, ReLU / Tanh, masks of 0 and 1, and batches that take the persistent loop round more than once; a guard fails when a
  served (family, N, configuration) has no case;
* the k-node gather (fm_gnn_gather) at E = 9, 17, 24, 35 and 64 under each mapping that serves E: bit for bit the k
  one-node calls of fm_gnn_forward side by side;
* batch invariance of the gather and of the wide head;
* RolloutCollector with each critic configuration at navigation N = 3 / O = 3, N = 7 / O = 3, N = 16 / O = 3 and formation
  N = 5 / O = 2: the actor and the env are untouched (bitwise the slabs, actions and log-probs of a collector with the
  default critic), stored values and finish() returns follow a float64 recomputation on the buffer's own slabs, the fused
  and dense collectors agree, and a captured episode replays bitwise as the eager one;
* a critic outside the fused family still runs through the collector on the dense path with cent_obs fed.
"""
import copy

import pytest
import torch

from test_gpu_policy import TOL, _assert_bar, _gnn, _perturb, _rel_err

pytestmark = pytest.mark.gpu

CONFIGS = {"cent_global": dict(use_cent_obs=True, critic_graph_aggr="global"),
           "node": dict(use_cent_obs=False, critic_graph_aggr="node"),
           "cent_node": dict(use_cent_obs=True, critic_graph_aggr="node")}
FAMILIES = {"navigation": dict(obs_dim=7, node_feat_dim=11, max_n=32), "formation": dict(obs_dim=11, node_feat_dim=13, max_n=7)}
ROWS_PER_ROUND = 148 * 16 * 8                  # SMs x warps per CTA x rows per warp tile: more rows go round again


def _cfg(family, N, config, **kw):
    import fair_marl_b200 as fm
    f = FAMILIES[family]
    return fm.PolicyConfig(num_agents=N, obs_dim=f["obs_dim"], node_feat_dim=f["node_feat_dim"], **CONFIGS[config], **kw)


def _head_cases():
    """(family, N, configuration, layer_N, recurrent, feature norm, ReLU, envs): every served triple once, the knobs
    cycling with different periods."""
    cases, i = [], 0
    for family, f in FAMILIES.items():
        for N in range(2, f["max_n"] + 1):
            for config in CONFIGS:
                B = (ROWS_PER_ROUND + 1000) // N + 1 if i % 5 == 0 else max(3, 1500 // N)
                cases.append((family, N, config, i % 3, (i // 3) % 2 == 0, (i // 2) % 2 == 0, (i // 4) % 2 == 0, B))
                i += 1
    return cases


HEAD_CASES = _head_cases()


def _critic(cfg, seed):
    import fair_marl_b200 as fm
    torch.manual_seed(seed)
    return _perturb(fm.DenseGraphCritic(cfg).eval().cuda(), skip="gnn_base.")


def _head_inputs(cfg, B, seed):
    N = cfg.num_agents
    M = B * N
    g = torch.Generator(device="cuda").manual_seed(seed)
    cent = 2 * torch.randn(B, N * cfg.obs_dim, generator=g, device="cuda") if cfg.use_cent_obs else None
    nbd = 2 * torch.randn(M, 16 * (N if cfg.critic_graph_aggr == "node" else 1), generator=g, device="cuda")
    rnn = torch.randn(M, 1, 64, generator=g, device="cuda")
    masks = (torch.rand(M, 1, generator=g, device="cuda") < 0.7).float()
    assert 0 < masks.sum() < M
    return cent, nbd, rnn, masks


def _reference(net, cent, nbd, rnn, masks, N):
    x = nbd if cent is None else torch.cat([cent.repeat_interleave(N, dim=0), nbd], dim=1)
    x, h = net.base(x), None
    if net.recurrent:
        x, h = net.rnn(x, rnn, masks)
    return net.v_out(x), h


@pytest.mark.parametrize("family,N,config,layer_N,recurrent,feat_norm,relu,B", HEAD_CASES)
def test_wide_critic_head_matches_float64(family, N, config, layer_N, recurrent, feat_norm, relu, B):
    cfg = _cfg(family, N, config, layer_N=layer_N, use_recurrent_policy=recurrent, use_feature_normalization=feat_norm,
               use_ReLU=relu)
    net = _critic(cfg, seed=N)
    assert net.critic_head_supported()
    cent, nbd, rnn, masks = _head_inputs(cfg, B, seed=N + 100)
    with torch.no_grad():
        v32, h32 = _reference(net, cent, nbd, rnn, masks, N)
        f64 = lambda x: None if x is None else x.double()
        v64, h64 = _reference(copy.deepcopy(net).double(), f64(cent), f64(nbd), f64(rnn), f64(masks), N)
        v, h = net._run_critic_head(None if cent is None else (cent, N), nbd, rnn, masks)
    _assert_bar(_rel_err(v, v64), _rel_err(v32, v64), "values")
    if recurrent:
        _assert_bar(_rel_err(h, h64), _rel_err(h32, h64), "rnn_out")
    else:
        assert h is rnn


def test_head_cases_cover_every_served_critic():
    """Every (family, N, configuration) whose graph network and head the fused kernels cover has a case; the head's
    input width D stays within the cap there, and the cap is refused one feature above."""
    from fair_marl_b200 import _lib
    import fair_marl_b200 as fm
    lib = _lib.load()
    have = {(c[0], c[1], c[2]) for c in HEAD_CASES}
    served = set()
    for family, f in FAMILIES.items():
        for N in range(2, 40):
            if family == "formation" and N > f["max_n"]:
                continue
            if not lib.fm_gnn_mapping(2 * N, f["node_feat_dim"]):        # the smallest graph of N agents: 2N entities
                continue
            for config in CONFIGS:
                net = fm.DenseGraphCritic(_cfg(family, N, config))
                if net.critic_head_supported():
                    served.add((family, N, config))
    assert served == have, (sorted(served - have), sorted(have - served))
    assert fm.DenseGraphCritic(_cfg("navigation", 32, "cent_node"))._head_in == 736
    assert ("navigation", 33, "node") not in served                     # 66 entities: no fused graph network


# ---- the k-node gather -------------------------------------------------------------------------------------------------
def _graph_inputs(B, rep, E, NF, seed, k):
    M = B * rep
    g = torch.Generator(device="cuda").manual_seed(seed)
    pos = torch.rand(B, E, 2, generator=g, device="cuda") * 2 - 1
    adj = torch.cdist(pos, pos).float().contiguous()
    node = torch.randn(M, E, NF, generator=g, device="cuda")
    node[..., -1] = torch.randint(0, 4, (M, E), generator=g, device="cuda").float()
    aid = torch.randint(0, E, (M, k), generator=g, device="cuda")
    aid[:, 0] = torch.arange(M, device="cuda") % rep                   # share_agent_id's first columns: the ego agents
    return adj, node, aid


def _mappings(E):
    from fair_marl_b200 import _lib
    return (1, 2) if _lib.load().fm_gnn_supported(E, 11) else (2,)


@pytest.mark.parametrize("E,k,rep", [(9, 3, 3), (9, 9, 3), (17, 7, 7), (24, 7, 7), (35, 16, 16), (35, 2, 16), (64, 32, 32),
                                     (64, 64, 1)])
def test_gather_equals_one_node_calls(E, k, rep):
    gnn = _gnn("node", E + k, node_feat_dim=11)
    adj, node, aid = _graph_inputs(700 // rep + 5, rep, E, 11, seed=E * k, k=k)
    with torch.no_grad():
        for mapping in _mappings(E):
            out = gnn.forward_fused(node, adj, rep, aid, mapping=mapping)
            assert out.shape == (node.shape[0], 16 * k)
            ones = torch.cat([gnn.forward_fused(node, adj, rep, aid[:, i:i + 1], mapping=mapping) for i in range(k)], dim=1)
            assert torch.equal(out, ones), (E, k, mapping)


@pytest.mark.parametrize("E,k,rep", [(9, 3, 3), (35, 16, 16), (64, 32, 32)])
def test_gather_is_batch_invariant(E, k, rep):
    gnn = _gnn("node", E, node_feat_dim=13)
    B = 2400 // rep + 7
    adj, node, aid = _graph_inputs(B, rep, E, 13, seed=E, k=k)
    M = node.shape[0]
    with torch.no_grad():
        for mapping in _mappings(E):
            full = gnn.forward_fused(node, adj, rep, aid, mapping=mapping)
            for m in (0, 1, M // 2, M - 1):
                alone = gnn.forward_fused(node[m:m + 1], adj[m // rep:m // rep + 1], 1, aid[m:m + 1], mapping=mapping)
                assert torch.equal(alone[0], full[m]), (m, mapping)
            k0 = 37
            part = gnn.forward_fused(node[k0 * rep:], adj[k0:], rep, aid[k0 * rep:], mapping=mapping)
            assert torch.equal(part, full[k0 * rep:])


@pytest.mark.parametrize("family,N,config", [("navigation", 3, "cent_global"), ("navigation", 16, "cent_node"),
                                             ("navigation", 32, "cent_node"), ("formation", 7, "node")])
def test_wide_critic_head_is_batch_invariant(family, N, config):
    net = _critic(_cfg(family, N, config), seed=3)
    B = ROWS_PER_ROUND // N + 123
    cent, nbd, rnn, masks = _head_inputs(net.cfg, B, seed=N)
    c = lambda lo, hi: None if cent is None else (cent[lo:hi], N)
    with torch.no_grad():
        full, hf = net._run_critic_head(c(0, B), nbd, rnn, masks)
        again, _ = net._run_critic_head(c(0, B), nbd, rnn, masks)
        assert torch.equal(full, again)
        for b in (0, 1, B // 2, B - 1):
            lo, hi = b * N, (b + 1) * N
            v, h = net._run_critic_head(c(b, b + 1), nbd[lo:hi], rnn[lo:hi], masks[lo:hi])
            assert torch.equal(v, full[lo:hi]) and torch.equal(h, hf[lo:hi]), b
        b0 = 37
        v, _ = net._run_critic_head(c(b0, B), nbd[b0 * N:], rnn[b0 * N:], masks[b0 * N:])
        assert torch.equal(v, full[b0 * N:])


# ---- the collector -----------------------------------------------------------------------------------------------------
SHAPES = [("navigation", 3, 3), ("navigation", 7, 3), ("navigation", 16, 3), ("formation", 5, 2)]


def _env(family, N, O, num_envs, episode_length=8, seed=11):
    import fair_marl_b200 as fm
    if family == "navigation":
        from oracle.navgraph import NavConfig
        from parity_util import sim_config_from
        return fm.B200GraphVecEnv(sim_config_from(NavConfig(num_agents=N, num_obstacles=O, episode_length=episode_length)),
                                  num_envs=num_envs, seed=seed)
    cfg = fm.FormationSimConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=episode_length)
    return fm.B200FormationVecEnv(cfg, num_envs=num_envs, seed=seed)


def _policy(family, N, config, scale, **critic_kw):
    import fair_marl_b200 as fm
    f = FAMILIES[family]
    torch.manual_seed(0)
    actor = fm.DenseGraphActor(fm.PolicyConfig(num_agents=N, obs_dim=f["obs_dim"], node_feat_dim=f["node_feat_dim"])).cuda().eval()
    with torch.no_grad():
        actor.action_out.weight.mul_(scale)
    ccfg = fm.PolicyConfig(num_agents=N, obs_dim=f["obs_dim"], node_feat_dim=f["node_feat_dim"],
                           **(CONFIGS[config] if config else {}), **critic_kw)
    torch.manual_seed(1)
    critic = _perturb(fm.DenseGraphCritic(ccfg).cuda().eval(), skip="gnn_base.")
    return actor, critic


def _collect(shape, config, *, deterministic=False, fused=None, capture=False, finish=False, **critic_kw):
    import fair_marl_b200 as fm
    family, N, O = shape
    env = _env(family, N, O, 48)
    actor, critic = _policy(family, N, config, 100.0 if deterministic else 20.0, **critic_kw)
    col = fm.RolloutCollector(env, actor, critic, deterministic=deterministic, fused=fused,
                              generator=torch.Generator(device=env.device).manual_seed(5))
    col.warmup(); col.run(); col.buffer.after_update()
    if capture:
        col.capture()
    col.run()
    if finish:
        col.finish()
    torch.cuda.synchronize()
    b = col.buffer
    env.close()
    return col, critic, b


def _float64_values(critic, b):
    """Values of every slab (0..T) recomputed by the dense critic in fp32 and in float64 from the buffer's own slabs, fed
    as GMPERunner.collect feeds GR_Critic: share_obs and share_agent_id."""
    T, B, N, E = b.episode_length, b.n_rollout_threads, b.num_agents, b.num_entities
    M = B * N
    ref = copy.deepcopy(critic).double()
    out32, out64 = [], []
    with torch.no_grad():
        for t in range(T + 1):
            cent = b.share_obs[t].reshape(M, -1)
            aid = b.share_agent_id[t].reshape(M, N) if critic.cfg.critic_graph_aggr == "node" else b.agent_id[t].reshape(M, 1)
            args = (cent, b.node_obs[t].view(M, E, -1), b.adj_env[t].repeat_interleave(N, 0), aid,
                    b.rnn_states_critic[t].view(M, 1, -1), b.masks[t].view(M, 1))
            out32.append(critic(*args)[0].view(B, N, 1))
            out64.append(ref(*[a.double() if a.is_floating_point() else a for a in args])[0].view(B, N, 1))
    return torch.stack(out32), torch.stack(out64)


def _returns64(b, v64):
    gae = torch.zeros_like(v64[0])
    ret = torch.zeros_like(v64)
    rw, mk = b.rewards.double(), b.masks.double()
    for t in reversed(range(b.episode_length)):
        delta = rw[t] + b.gamma * v64[t + 1] * mk[t + 1] - v64[t]
        gae = delta + b.gamma * b.gae_lambda * mk[t + 1] * gae
        ret[t] = gae + v64[t]
    return ret


@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}-N{s[1]}-O{s[2]}")
def test_collector_with_critic(shape, config):
    col, critic, b = _collect(shape, config, finish=True)
    assert col.fused
    _, _, b0 = _collect(shape, None)                                  # the default critic, same seeds
    for name in ("obs", "node_obs", "adj_env", "rewards", "dones", "actions_env", "action_log_probs", "rnn_states", "masks"):
        assert torch.equal(getattr(b, name), getattr(b0, name)), name
    T = b.episode_length
    v32, v64 = _float64_values(critic, b)
    _assert_bar(_rel_err(b.value_preds[:T], v64[:T]), _rel_err(v32[:T], v64[:T]), "stored values")
    _assert_bar(_rel_err(b.value_preds[T], v64[T]), _rel_err(v32[T], v64[T]), "bootstrap value")
    r64 = _returns64(b, v64)
    r32 = _returns64(b, v32.double())
    _assert_bar(_rel_err(b.returns[:T], r64[:T]), _rel_err(r32[:T].float(), r64[:T]), "returns")
    # a captured episode replays bitwise as the eager one
    _, _, bg = _collect(shape, config, capture=True, finish=True)
    for name in ("obs", "node_obs", "adj_env", "actions_env", "action_log_probs", "rnn_states", "rnn_states_critic",
                 "value_preds", "returns"):
        assert torch.equal(getattr(b, name), getattr(bg, name)), name


@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}-N{s[1]}-O{s[2]}")
def test_collector_fused_and_dense_agree(shape, config):
    colf, critic, bf = _collect(shape, config, deterministic=True, finish=True)
    cold, _, bd = _collect(shape, config, deterministic=True, fused=False, finish=True)
    assert colf.fused and not cold.fused
    assert torch.equal(bf.actions_env, bd.actions_env) and torch.equal(bf.obs, bd.obs)
    T = bf.episode_length
    _, v64 = _float64_values(critic, bf)
    _assert_bar(_rel_err(bf.value_preds, v64), _rel_err(bd.value_preds, v64), "fused vs dense values")
    r64 = _returns64(bf, v64)
    _assert_bar(_rel_err(bf.returns[:T], r64[:T]), _rel_err(bd.returns[:T], r64[:T]), "fused vs dense returns")


def test_critic_outside_the_fused_family_runs_dense_with_cent_obs():
    """layer_N = 3 is outside both fused heads: the collector still goes fused for the actor, and the critic falls back to
    the dense modules with share_obs fed as rows."""
    shape = ("navigation", 3, 3)
    col, critic, b = _collect(shape, "cent_node", finish=True, layer_N=3)
    assert col.fused and not critic.critic_head_supported()
    T = b.episode_length
    v32, v64 = _float64_values(critic, b)
    _assert_bar(_rel_err(b.value_preds[:T], v64[:T]), _rel_err(v32[:T], v64[:T]), "dense-path values")
