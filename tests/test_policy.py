"""Dense graph policy (fair_marl_b200.policy) vs the reference's GR_Actor / GR_Critic.

* golden: outputs of the UNMODIFIED reference policy code (run from its checkout on the torch_geometric
  stand-in, oracle/make_policy_golden.py) -- state dict, inputs and outputs frozen in tests/golden/policy_*.npz;
* live (``-m reference``, only where FAIRMARL_REFERENCE_ROOT names the original project's checkout): fresh random
  configurations against the reference modules, and the shipped ``model_weights/*/actor.pt`` (legacy gnn.py key layout) loaded strictly.
Tolerance: 1e-5 * max(|ref|, 1) on float32 outputs (the contract of north_star); actions (argmax) exact.
"""
import ast
import glob
import os
from argparse import Namespace

import numpy as np
import pytest
import torch

from fair_marl_b200.policy import (DenseGraphActor, DenseGraphCritic, PolicyConfig, config_from_state_dict, edge_mask,
                                   load_reference_state_dict)
from oracle import reference_shim

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
TOL = 1e-5


def close(a, b, tol=TOL):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.all(np.abs(a - b) <= tol * np.maximum(np.abs(b), 1.0)), float(np.max(np.abs(a - b)))


def _cfg(N, overrides):
    from oracle.make_policy_golden import BASE_ARGS
    return PolicyConfig.from_args(Namespace(**{**BASE_ARGS, "num_agents": N, **overrides}))


def _flat(a):
    return torch.as_tensor(a.reshape((-1,) + a.shape[2:]))


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "policy_*.npz"))), ids=os.path.basename)
def test_policy_matches_reference_golden(path):
    z = np.load(path)
    N, O, B, _ = (int(v) for v in z["meta"])
    E = 2 * N + O
    cfg = _cfg(N, ast.literal_eval(str(z["overrides"])))
    actor, critic = DenseGraphActor(cfg).eval(), DenseGraphCritic(cfg).eval()
    load_reference_state_dict(actor, {k[6:]: z[k] for k in z.files if k.startswith("actor/")})
    load_reference_state_dict(critic, {k[7:]: z[k] for k in z.files if k.startswith("critic/")})
    # the env's distance matrix, shared by its N agents, as a stride-0 view (what the simulator hands over)
    adj = torch.as_tensor(z["in_adj_env"])[:, None].expand(B, N, E, E).reshape(B * N, E, E)
    obs, node, aid = _flat(z["in_obs"]), _flat(z["in_node_obs"]), _flat(z["in_agent_id"])
    rnn, masks = _flat(z["in_rnn_states"]), _flat(z["in_masks"])
    with torch.no_grad():
        act, logp, h = actor(obs, node, adj, aid, rnn, masks, deterministic=True)
        feat = actor.gnn_base(node, adj, aid)
        val, hc = critic(None, node, adj, aid, rnn, masks)
    assert np.array_equal(act.numpy(), z["out_actions"])
    for name, got in (("gnn_feat", feat), ("action_log_probs", logp), ("rnn_out", h), ("values", val), ("rnn_out_critic", hc)):
        ok, err = close(got.numpy(), z["out_" + name])
        assert ok, (name, err)


def test_edge_mask_is_process_adj_connectivity():
    adj = torch.tensor([[0.0, 0.5, 1.0], [0.5, 0.0, 1.5], [1.0, 1.5, 0.0]])
    m = edge_mask(adj, 1.0)
    assert m.tolist() == [[False, True, False], [True, False, False], [False, False, False]]   # strict <, > 0


def test_sampling_is_a_valid_categorical_draw():
    cfg = PolicyConfig()
    actor = DenseGraphActor(cfg).eval()
    M, E = 64, 9
    g = torch.Generator().manual_seed(0)
    obs, node = torch.randn(M, 7, generator=g), torch.randn(M, E, 11, generator=g)
    node[..., -1] = torch.randint(0, 3, (M, E), generator=g).float()
    adj = torch.rand(M, E, E, generator=g) * 2
    with torch.no_grad():
        a, lp, h = actor(obs, node, adj, torch.zeros(M, 1, dtype=torch.long), torch.zeros(M, 1, 64), torch.ones(M, 1),
                         generator=torch.Generator().manual_seed(1))
    assert a.shape == (M, 1) and a.dtype == torch.int64 and int(a.min()) >= 0 and int(a.max()) < 5
    assert lp.shape == (M, 1) and torch.all(lp <= 0) and h.shape == (M, 1, 64)


needs_reference = pytest.mark.reference


@needs_reference
@pytest.mark.parametrize("N,O,over", [
    (3, 3, {}),
    (5, 0, dict(gnn_concat_heads=True, gnn_num_heads=2, use_feature_normalization=True, embed_layer_N=2)),
    (16, 3, dict(actor_graph_aggr="global", global_aggr_type="add", use_recurrent_policy=False)),
])
def test_policy_matches_live_reference(N, O, over):
    from oracle.make_policy_golden import BASE_ARGS, reference_policy, run_reference, synthetic_inputs
    args = Namespace(**{**BASE_ARGS, "num_agents": N, **over})
    ref_actor, ref_critic = reference_policy(args, 2 * N + O, seed=7)
    x = synthetic_inputs(5, N, O, args.hidden_size, seed=7)
    y = run_reference(ref_actor, ref_critic, x, N)
    cfg = PolicyConfig.from_args(args)
    actor, critic = DenseGraphActor(cfg).eval(), DenseGraphCritic(cfg).eval()
    load_reference_state_dict(actor, ref_actor.state_dict())
    load_reference_state_dict(critic, ref_critic.state_dict())
    f = lambda k: _flat(x[k])
    with torch.no_grad():
        act, logp, h = actor(f("obs"), f("node_obs"), f("adj"), f("agent_id"), f("rnn_states"), f("masks"), deterministic=True)
        val, hc = critic(None, f("node_obs"), f("adj"), f("agent_id"), f("rnn_states"), f("masks"))
    assert np.array_equal(act.numpy(), y["actions"])
    for name, got in (("action_log_probs", logp), ("rnn_out", h), ("values", val)):
        ok, err = close(got.numpy(), y[name])
        assert ok, (name, err)


@needs_reference
@pytest.mark.parametrize("variant", ["FA", "FA+FR", "RA", "OA"])
def test_shipped_actor_weights_load_strictly(variant):
    """model_weights/*/actor.pt use the legacy gnn.py EmbedConv key layout (lin1.0 / lin2.i.0) and the formation
    family's shapes (13 node features, 11-dim obs); they must load strictly and drive a forward pass."""
    path = os.path.join(reference_shim.REFERENCE_ROOT, "model_weights", variant, "actor.pt")
    sd = torch.load(path, map_location="cpu", weights_only=False)
    cfg = config_from_state_dict(sd)
    assert (cfg.node_feat_dim, cfg.obs_dim, cfg.gnn_num_heads, cfg.gnn_layer_N) == (13, 11, 3, 2)
    actor = DenseGraphActor(cfg).eval()
    load_reference_state_dict(actor, sd)
    # legacy EmbedConv of the reference, same weights, edge-list path
    from oracle import pyg_stub
    reference_shim.install_stubs(); pyg_stub.install()
    from onpolicy.algorithms.utils.gnn import EmbedConv
    ref = EmbedConv(input_dim=12, num_embeddings=4, embedding_size=2, hidden_size=16, layer_N=1, use_orthogonal=True,
                    use_ReLU=False, use_layerNorm=True, add_self_loop=False, edge_dim=1)
    use_relu = False
    try:
        ref.load_state_dict({k[len("gnn_base.gnn.embed_layer."):]: v for k, v in sd.items() if "embed_layer" in k})
    except RuntimeError:
        pytest.skip("legacy EmbedConv signature differs")
    g = torch.Generator().manual_seed(3)
    M, E = 4, 9
    x = torch.randn(M, E, 13, generator=g); x[..., -1] = torch.randint(0, 3, (M, E), generator=g).float()
    adj = torch.rand(M, E, E, generator=g) * 1.6; adj = (adj + adj.transpose(1, 2)) / 2; adj[:, range(E), range(E)] = 0
    m = edge_mask(adj, 1.0)
    idx = m.nonzero()
    ei = torch.stack([idx[:, 0] * E + idx[:, 1], idx[:, 0] * E + idx[:, 2]])
    ea = adj[idx[:, 0], idx[:, 1], idx[:, 2]].unsqueeze(1)
    cfg_act = PolicyConfig(**{**cfg.__dict__, "embed_use_ReLU": use_relu})
    dense = DenseGraphActor(cfg_act).eval(); load_reference_state_dict(dense, sd)
    with torch.no_grad():
        want = ref(x.view(-1, 13), ei, ea).view(M, E, -1)
        got = dense.gnn_base.embed_layer(x, adj, m)
    ok, err = close(got.numpy(), want.numpy())
    assert ok, err
