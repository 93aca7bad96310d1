"""``-m reference``: the dense critic (fair_marl_b200.policy.DenseGraphCritic) with use_cent_obs=True and with
critic_graph_aggr='node' against the live reference GR_Critic, fed share_obs and share_agent_id as
graph_MAPPOPolicy.get_actions feeds it (GMPERunner.collect: cent_obs = share_obs, agent_id = share_agent_id for the
critic).  The dense modules are the oracle of the fused critic kernels (tests/critic_cent), so this pins those kernels to
the reference too.  Skips where there is no reference checkout (FAIRMARL_REFERENCE_ROOT)."""
from argparse import Namespace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.reference


@pytest.mark.parametrize("N,O,over", [
    (3, 3, dict(use_cent_obs=True)),
    (3, 3, dict(critic_graph_aggr="node")),
    (7, 3, dict(use_cent_obs=True, critic_graph_aggr="node", use_recurrent_policy=False, layer_N=2)),
    (16, 3, dict(use_cent_obs=True, critic_graph_aggr="node")),
])
def test_dense_critic_matches_live_reference(N, O, over):
    from fair_marl_b200.policy import DenseGraphCritic, PolicyConfig, load_reference_state_dict
    from oracle.make_policy_golden import BASE_ARGS, reference_policy, synthetic_inputs
    args = Namespace(**{**BASE_ARGS, "num_agents": N, **over})
    _, ref_critic = reference_policy(args, 2 * N + O, seed=3)
    x = synthetic_inputs(4, N, O, args.hidden_size, seed=3)
    B = x["obs"].shape[0]
    flat = lambda a: torch.as_tensor(np.ascontiguousarray(a.reshape((-1,) + a.shape[2:])))
    share_obs = np.repeat(x["obs"].reshape(B, 1, -1), N, axis=1)                       # graph_mpe_runner.py:470-473
    share_agent_id = np.repeat(x["agent_id"].reshape(B, 1, N), N, axis=1)
    aid = share_agent_id if args.critic_graph_aggr == "node" else x["agent_id"]
    args_in = (flat(share_obs), flat(x["node_obs"]), flat(x["adj"]), flat(aid), flat(x["rnn_states"]), flat(x["masks"]))
    critic = DenseGraphCritic(PolicyConfig.from_args(args)).eval()
    load_reference_state_dict(critic, ref_critic.state_dict())
    with torch.no_grad():
        want, want_h = ref_critic(*args_in)
        got, got_h = critic(*args_in)
    for a, b in ((got, want), (got_h, want_h)):
        a, b = a.numpy().astype(np.float64), b.numpy().astype(np.float64)
        assert np.all(np.abs(a - b) <= 1e-5 * np.maximum(np.abs(b), 1.0)), float(np.abs(a - b).max())
