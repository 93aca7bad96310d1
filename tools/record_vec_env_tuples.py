"""Record what ``B200GraphVecEnv`` hands to the runner -- the reset 4-tuple and a few step 7-tuples, exactly as returned
(shapes, dtypes, the infos sequence) -- for tests/test_reference_runner.py, which replays them through the UNMODIFIED
GMPERunner from a checkout of the original project (FAIRMARL_REFERENCE_ROOT), which needs no GPU.
usage (GPU box): python tools/record_vec_env_tuples.py gpurun_out/b200_vec_env_tuples.npz"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

import fair_marl_b200 as fm

B, N, O, T = 6, 3, 3, 7
cfg = fm.SimConfig(num_agents=N, num_obstacles=O, episode_length=5, goal_rew=30.0, collision_rew=30.0, info_every_step=True)
env = fm.B200GraphVecEnv(cfg, num_envs=B, seed=3)
out = {"meta": np.array([B, N, O, T, cfg.episode_length])}
for k, a in zip(("obs", "agent_id", "node_obs", "adj"), env.reset(copy=True)):
    out["reset_" + k] = np.array(a)
rng = np.random.default_rng(0)
eye = np.eye(5, dtype=np.float32)
for t in range(T):
    act = eye[rng.integers(0, 5, (B, N))]
    obs, ag, node, adj, rew, done, infos = env.step(act, copy=True)
    out[f"step{t}_actions"] = act
    for k, a in zip(("obs", "agent_id", "node_obs", "adj", "rewards", "dones"), (obs, ag, node, adj, rew, done)):
        out[f"step{t}_{k}"] = np.array(a)
    assert len(infos) == B and len(infos[0]) == N and isinstance(infos[0][0], dict)
    out[f"step{t}_info_keys"] = np.array(list(infos[0][0].keys()))
    out[f"step{t}_infos"] = np.array([[[infos[b][i][k] for k in infos[b][i]] for i in range(N)] for b in range(B)], dtype=np.float32)
env.close()
path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "gpurun_out", "b200_vec_env_tuples.npz")
os.makedirs(os.path.dirname(path), exist_ok=True)
np.savez_compressed(path, **out)
print("wrote", path, {k: (v.shape, str(v.dtype)) for k, v in out.items() if k.startswith(("reset_", "step0_"))})
