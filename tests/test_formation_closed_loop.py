"""End-to-end semantic check of the widened rows together (SURVEY.md section 8f, N2 x N3), on the CPU: the actors the
reference SHIPS (model_weights/{FA+FR,FA,OA,RA}/actor.pt, trained on the formation scenarios) are loaded into
fair_marl_b200's dense GNN policy and drive the formation oracle in closed loop.  If any piece of the interface were off --
the 11-dim observation, the 13-dim node rows, adj, the agent-id gather, the 0..4 action convention, the per-scenario goal
semantics -- a trained policy would do no better than random moves.  Needs the original project's checkout (the weights live
there): FAIRMARL_REFERENCE_ROOT."""
import os

import numpy as np
import pytest
import torch

from oracle import reference_shim
from oracle.formation import FormationConfig, FormationOracle

SCENARIO = {"FA+FR": ("fair", True), "FA": ("fair", False), "OA": ("optimal", False), "RA": ("random", False)}


def _rollout(variant: str, use_policy: bool, B: int = 16, steps: int = 50, seed: int = 3):
    from fair_marl_b200.policy import DenseGraphActor, config_from_state_dict, load_reference_state_dict
    mode, fair = SCENARIO[variant]
    cfg = FormationConfig(num_agents=3, num_obstacles=3, goal_rew=30.0, collision_rew=30.0, assignment=mode,
                          fairness_reward=fair)                       # model_weights/*/config.yaml
    N, E = cfg.num_agents, cfg.num_entities
    orc = FormationOracle(cfg, B, seed=seed)
    o = orc.reset()
    rng = np.random.default_rng(seed)
    if use_policy:
        sd = torch.load(os.path.join(reference_shim.REFERENCE_ROOT, "model_weights", variant, "actor.pt"),
                        map_location="cpu", weights_only=False)
        pc = config_from_state_dict(sd)
        actor = DenseGraphActor(pc).eval()
        load_reference_state_dict(actor, sd)
        rnn = torch.zeros(B * N, pc.recurrent_N, pc.hidden_size)
        masks = torch.ones(B * N, 1)
        agent_id = torch.arange(N).repeat(B).view(B * N, 1).float()
    total = 0.0
    for t in range(steps):
        if use_policy:
            obs = torch.tensor(o["obs"], dtype=torch.float32).view(B * N, -1)
            node = torch.tensor(o["node_obs"], dtype=torch.float32).view(B * N, E, -1)
            adj = torch.tensor(o["adj"], dtype=torch.float32).unsqueeze(1).expand(B, N, E, E).reshape(B * N, E, E)
            with torch.no_grad():
                a, _, rnn = actor(obs, node, adj, agent_id, rnn, masks, deterministic=True)
            a = a.view(B, N).numpy()
        else:
            a = rng.integers(0, 5, (B, N))
        o = orc.step(a)
        total += float(o["reward"].mean())
        if use_policy:
            masks = torch.tensor(1.0 - o["done"].astype(np.float32)).view(B * N, 1)
    return total / steps, orc.branch_hits.get("status_latched", 0)


@pytest.mark.reference
@pytest.mark.parametrize("variant", sorted(SCENARIO))
def test_shipped_actor_reaches_goals_on_our_observations(variant):
    rew_p, latched_p = _rollout(variant, True)
    rew_r, latched_r = _rollout(variant, False)
    assert latched_p >= 20 and latched_p >= 5 * max(latched_r, 1), (variant, latched_p, latched_r)
    assert rew_p > rew_r + 0.3, (variant, rew_p, rew_r)          # FA+FR carries the (mostly negative) fairness term
