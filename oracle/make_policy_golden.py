"""Golden vectors for the dense graph policy (TEST INFRASTRUCTURE ONLY; needs FAIRMARL_REFERENCE_ROOT).

Builds the UNMODIFIED reference ``GR_Actor`` / ``GR_Critic`` (onpolicy/algorithms/graph_actor_critic.py) on top of
the ``gym`` stub (reference_shim) and the torch_geometric stand-in (pyg_stub), feeds them seeded inputs shaped like
the simulator's outputs (distances with isolated nodes, one adjacency per env shared by its agents) and records
state dict + inputs + outputs to ``tests/golden/policy_*.npz``.

    python -m oracle.make_policy_golden
"""
from __future__ import annotations

import os
from argparse import Namespace

import numpy as np
import torch

from . import pyg_stub, reference_shim

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

BASE_ARGS = dict(
    hidden_size=64, gain=0.01, use_orthogonal=True, use_policy_active_masks=True, use_naive_recurrent_policy=False,
    use_recurrent_policy=True, recurrent_N=1, gnn_hidden_size=16, gnn_num_heads=3, gnn_concat_heads=False,
    num_embeddings=4, embedding_size=2, gnn_layer_N=2, gnn_use_ReLU=True, actor_graph_aggr="node",
    critic_graph_aggr="global", global_aggr_type="mean", embed_hidden_size=16, embed_layer_N=1, embed_use_ReLU=True,
    use_feature_normalization=True, embed_add_self_loop=False, max_edge_dist=1.0, use_ReLU=True, stacked_frames=1,
    layer_N=1, use_popart=False, use_cent_obs=False, num_agents=3, split_batch=False, max_batch_size=32)


def reference_policy(args: Namespace, num_entities: int, obs_dim: int = 7, node_feat: int = 11, seed: int = 0):
    """(GR_Actor, GR_Critic) of the reference, freshly initialised with ``seed``."""
    reference_shim.install_stubs()
    pyg_stub.install()
    import gym
    from onpolicy.algorithms.graph_actor_critic import GR_Actor, GR_Critic
    Box, Disc = gym.spaces.Box, gym.spaces.Discrete
    torch.manual_seed(seed)
    actor = GR_Actor(args, Box(0, 0, (obs_dim,)), Box(0, 0, (num_entities, node_feat)), Box(0, 0, (1,)), Disc(5))
    critic = GR_Critic(args, Box(0, 0, (obs_dim * args.num_agents,)), Box(0, 0, (num_entities, node_feat)), Box(0, 0, (1,)))
    # LayerNorm / bias parameters start at 1 / 0 in the reference; perturb them so that the fixture pins them too
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for mod in (actor, critic):
            for name, prm in mod.named_parameters():
                if prm.dim() == 1:
                    prm.add_(0.1 * torch.randn(prm.shape, generator=g))
                if name.endswith("action_out.linear.weight"):
                    prm.mul_(50.0)                   # gain 0.01 leaves the logits nearly flat
    return actor.eval(), critic.eval()


def synthetic_inputs(B: int, N: int, O: int, hidden: int, seed: int):
    """Inputs with the simulator's structure: positions in the 2x2 world, ego-relative node features, one distance
    matrix per env (shared by its N agents), some far-away entities (isolated nodes at max_edge_dist = 1)."""
    rng = np.random.default_rng(seed)
    E = 2 * N + O
    pos = rng.uniform(-1, 1, (B, E, 2)).astype(np.float32)
    pos[:, -1] += 5.0 * (rng.random((B, 1)) < 0.3)                     # some isolated last entities
    vel = np.zeros((B, E, 2), np.float32)
    vel[:, :N] = rng.normal(0, 0.5, (B, N, 2))
    goal = pos.copy()
    goal[:, :N] = pos[:, N:2 * N][np.arange(B)[:, None], np.argsort(rng.random((B, N)), axis=1)]
    typ = np.concatenate([np.zeros(N), np.ones(N), 2 * np.ones(O)]).astype(np.float32)
    d = np.linalg.norm(pos[:, :, None].astype(np.float64) - pos[:, None].astype(np.float64), axis=-1).astype(np.float32)
    node = np.zeros((B, N, E, 11), np.float32)
    for a in range(N):
        rp = pos - pos[:, a:a + 1]
        node[:, a, :, 0:2] = vel - vel[:, a:a + 1]
        node[:, a, :, 2:4] = rp
        node[:, a, :, 4:6] = goal - pos[:, a:a + 1]
        node[:, a, :, 6:8] = rp
        node[:, a, :, 8:10] = rp
        node[:, a, :, 10] = typ
    obs = np.concatenate([vel[:, :N], pos[:, :N], goal[:, :N] - pos[:, :N], rng.normal(0, 1, (B, N, 1))], axis=-1).astype(np.float32)
    agent_id = np.tile(np.arange(N)[None, :, None], (B, 1, 1)).astype(np.int64)
    rnn = rng.normal(0, 0.3, (B, N, 1, hidden)).astype(np.float32)
    masks = (rng.random((B, N, 1)) > 0.2).astype(np.float32)
    adj = np.broadcast_to(d[:, None], (B, N, E, E)).copy()
    return dict(obs=obs, node_obs=node, adj=adj, adj_env=d, agent_id=agent_id, rnn_states=rnn, masks=masks)


def run_reference(actor, critic, x, N: int):
    flat = lambda a: torch.as_tensor(a.reshape((-1,) + a.shape[2:]))
    B = x["obs"].shape[0]
    share = np.repeat(x["obs"].reshape(B, 1, -1), N, axis=1)
    with torch.no_grad():
        act, logp, h = actor(flat(x["obs"]), flat(x["node_obs"]), flat(x["adj"]), flat(x["agent_id"]),
                             flat(x["rnn_states"]), flat(x["masks"]), deterministic=True)
        feat = actor.gnn_base(flat(x["node_obs"]), flat(x["adj"]), flat(x["agent_id"]))
        val, hc = critic(flat(share), flat(x["node_obs"]), flat(x["adj"]), flat(x["agent_id"]), flat(x["rnn_states"]), flat(x["masks"]))
    return dict(actions=act.numpy(), action_log_probs=logp.numpy(), rnn_out=h.numpy(), gnn_feat=feat.numpy(),
                values=val.numpy(), rnn_out_critic=hc.numpy())


def make(name: str, N: int, O: int, B: int, seed: int, **overrides):
    args = Namespace(**{**BASE_ARGS, "num_agents": N, **overrides})
    actor, critic = reference_policy(args, 2 * N + O, seed=seed)
    x = synthetic_inputs(B, N, O, args.hidden_size, seed)
    y = run_reference(actor, critic, x, N)
    blob = {"in_" + k: v for k, v in x.items() if k != "adj"}
    blob.update({"out_" + k: v for k, v in y.items()})
    blob.update({"actor/" + k: v.numpy() for k, v in actor.state_dict().items()})
    blob.update({"critic/" + k: v.numpy() for k, v in critic.state_dict().items()})
    blob["meta"] = np.array([N, O, B, seed])
    blob["overrides"] = np.array(repr(overrides))
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    np.savez_compressed(os.path.join(GOLDEN_DIR, f"policy_{name}.npz"), **blob)
    print(name, {k: v.shape for k, v in y.items()})


if __name__ == "__main__":
    make("n3_o3", 3, 3, 16, 0)
    make("n7_o3_concat_tanh", 7, 3, 6, 1, gnn_concat_heads=True, gnn_use_ReLU=False, use_ReLU=False, embed_use_ReLU=False,
         embed_layer_N=2, layer_N=2, gnn_layer_N=1, global_aggr_type="max")
