"""Drop-in proof with the reference's OWN runner (SURVEY.md section 8b / 8d C5; needs FAIRMARL_REFERENCE_ROOT).

The unmodified ``GMPERunner`` (onpolicy/runner/shared/graph_mpe_runner.py) is instantiated on top of what
``B200GraphVecEnv`` returns -- ``tests/golden/b200_vec_env_tuples.npz``, the reset 4-tuple and step 7-tuples recorded
from the device env on a B200 by tools/record_vec_env_tuples.py (the original project runs on the CPU from its own
checkout, so the hand-over is a recording) -- behind the same spaces object the device env builds
(``fair_marl_b200.vec_env.make_spaces``).  Then, with the reference's own code and nothing of ours in between:
``warmup`` (:178-203) -> per step ``collect`` (:396-436, the reference's GR_Actor / GR_Critic on its GraphReplayBuffer
slabs) -> ``envs.step(actions_env)`` -> the data tuple of ``run`` (:60-80) -> ``insert`` (:438-488), and finally
``compute`` (:490-506) and the info aggregation ``process_infos`` (base_runner.py:197-276).  Every slab of the
reference buffer must hold exactly what the env returned.  wandb / imageio / tensorboardX / torch_geometric are absent
here and stubbed in ``sys.modules`` (SURVEY.md Appendix A); they are not on the env path."""
import os
import sys
import types
from pathlib import Path

import numpy as np
import pytest

from oracle import reference_shim

pytestmark = pytest.mark.reference
FIXTURE = os.path.join(os.path.dirname(__file__), "golden", "b200_vec_env_tuples.npz")


class ReplayVecEnv:
    """Hands the recorded tuples to the runner one call at a time, with the attributes ``GraphSubprocVecEnv`` has."""

    def __init__(self, z):
        from fair_marl_b200.vec_env import make_spaces
        self.z = z
        self.B, self.N, self.O, self.T, _ = (int(v) for v in z["meta"])
        self.num_envs, self.t = self.B, 0
        for name, spaces in make_spaces(self.N, 2 * self.N + self.O).items():
            setattr(self, name, spaces)
        self.actions_seen = []

    def reset(self):
        return tuple(self.z["reset_" + k] for k in ("obs", "agent_id", "node_obs", "adj"))

    def step(self, actions_env):
        a = np.asarray(actions_env)
        assert a.shape == (self.B, self.N, 5) and np.all(a.sum(-1) == 1)     # one-hot rows, as graph_mpe_runner.py:429-431 builds them
        self.actions_seen.append(a)
        t, z = self.t, self.z
        self.t += 1
        keys = [str(k) for k in z[f"step{t}_info_keys"]]
        infos = [[{k: float(z[f"step{t}_infos"][b, i, j]) for j, k in enumerate(keys)} for i in range(self.N)] for b in range(self.B)]
        return tuple(z[f"step{t}_{k}"] for k in ("obs", "agent_id", "node_obs", "adj", "rewards", "dones")) + (infos,)

    def close(self):
        pass


def _stub_modules():
    from oracle import pyg_stub
    reference_shim.install_stubs()
    pyg_stub.install()
    for name in ("wandb", "imageio"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    if "tensorboardX" not in sys.modules:
        m = types.ModuleType("tensorboardX")

        class SummaryWriter:
            def __init__(self, *a, **k):
                pass

            def add_scalars(self, *a, **k):
                pass

            def close(self):
                pass
        m.SummaryWriter = SummaryWriter
        sys.modules["tensorboardX"] = m


@pytest.mark.skipif(not os.path.isfile(FIXTURE), reason="tests/golden/b200_vec_env_tuples.npz not recorded yet (tools/record_vec_env_tuples.py on a GPU box)")
def test_unmodified_gmpe_runner_consumes_the_device_env(tmp_path):
    import torch
    _stub_modules()
    z = np.load(FIXTURE)
    envs = ReplayVecEnv(z)
    B, N, O, T = envs.B, envs.N, envs.O, envs.T
    sys.argv = ["train_mpe.py"]
    from onpolicy.config import get_config, graph_config
    args, parser = graph_config([], get_config())                           # what train_mpe.py:109-114 does for GraphMPE
    args.env_name, args.algorithm_name, args.scenario_name = "GraphMPE", "rmappo", "navigation_graph"
    args.num_agents, args.num_obstacles, args.n_rollout_threads, args.episode_length = N, O, B, T
    args.use_wandb, args.use_render, args.model_dir, args.use_centralized_V = False, False, None, True
    args.num_mini_batch, args.ppo_epoch, args.use_valuenorm, args.use_popart = 1, 1, True, False
    from onpolicy.runner.shared.graph_mpe_runner import GMPERunner
    torch.manual_seed(0)
    runner = GMPERunner({"all_args": args, "envs": envs, "eval_envs": None, "device": torch.device("cpu"), "num_agents": N,
                         "run_dir": Path(tmp_path)})
    buf = runner.buffer
    runner.warmup()                                                           # graph_mpe_runner.py:178-203
    for k in ("obs", "node_obs", "adj", "agent_id"):
        assert np.array_equal(getattr(buf, k)[0], z["reset_" + k].astype(getattr(buf, k).dtype)), k
    all_infos = []
    for step in range(T):
        values, actions, logp, rnn, rnn_c, actions_env = runner.collect(step)              # :396-436
        obs, agent_id, node_obs, adj, rewards, dones, infos = envs.step(actions_env)
        assert actions_env.shape == (B, N, 5) and dones.dtype == np.bool_ and rewards.shape == (B, N)
        rewards = rewards[:, :, np.newaxis]                                                # :76
        available = np.ones((B, N, 5), dtype=np.float32)
        runner.insert((obs, agent_id, node_obs, adj, agent_id, rewards, dones, infos, values, actions, logp, rnn, rnn_c, available))   # :438-488
        all_infos.append(infos)
        for k, got in (("obs", obs), ("node_obs", node_obs), ("adj", adj), ("agent_id", agent_id)):
            assert np.array_equal(getattr(buf, k)[step + 1], got.astype(getattr(buf, k).dtype)), (step, k)
        assert np.array_equal(buf.rewards[step], rewards) and np.array_equal(buf.masks[step + 1][..., 0], 1.0 - dones)
        assert np.array_equal(buf.share_obs[step + 1][:, 0], obs.reshape(B, -1))           # centralized V: all agents' obs side by side
    runner.compute()                                                                       # :490-506 (bootstrap value, returns)
    assert np.isfinite(buf.returns).all() and np.isfinite(buf.value_preds).all()
    env_infos = runner.process_infos(all_infos[-1])                                        # base_runner.py:197-276
    assert any("individual_rewards" in k or "individual_reward" in k for k in env_infos) and len(env_infos) > 0
    train_infos = runner.train()                                                           # one PPO update on the collected slabs
    assert all(np.isfinite(v) for v in train_infos.values() if isinstance(v, (int, float, np.floating)))
    assert runner.buffer.step == 0 and len(envs.actions_seen) == T


def test_spaces_match_the_reference_env():
    """The spaces object of the device env (make_spaces) against the unmodified GraphMPE env's, shape by shape."""
    from fair_marl_b200.vec_env import make_spaces
    from oracle.navgraph import NavConfig
    env, _ = reference_shim.make_reference_env(NavConfig(num_agents=3, num_obstacles=3))
    ours = make_spaces(3, 9)
    for name in ("observation_space", "share_observation_space", "node_observation_space", "adj_observation_space",
                 "edge_observation_space", "agent_id_observation_space", "share_agent_id_observation_space"):
        ref = getattr(env, name)
        assert len(ref) == len(ours[name]) == 3
        for r, o in zip(ref, ours[name]):
            assert tuple(r.shape) == tuple(o.shape) and o.__class__.__name__ == "Box", name
    for r, o in zip(env.action_space, ours["action_space"]):
        assert r.n == o.n == 5 and o.__class__.__name__ == "Discrete"
