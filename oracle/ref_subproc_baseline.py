"""The reference's own CPU path, timed as SURVEY.md section 8(d) / BASELINE.md section 3 specify: the UNMODIFIED
``GraphSubprocVecEnv`` (onpolicy/envs/env_wrappers.py:951-1025) over the unmodified ``GraphMPEEnv`` / ``MultiAgentGraphEnv`` +
``navigation_graph.Scenario``, one worker process per env, random one-hot actions, episode_length 25 with auto-reset.
TEST / MEASUREMENT INFRASTRUCTURE ONLY; needs the original project's checkout (FAIRMARL_REFERENCE_ROOT), not a GPU: its
JSON lines are committed under profiles/ next to the port's numbers (bench.py cpu_baseline, kind "port").

Gurobi / pyomo are not installable (requirements.txt:2), so the assignment solver is stubbed and the stub is stated:
  bruteforce  lexicographic-min over permutations (cheapest: favours the CPU path)
  highs       the reference's iterated MILP restated on scipy.optimize.milp (closest in kind to gurobi_persistent)

usage: python -m oracle.ref_subproc_baseline [--envs N ...] [--agents 3] [--steps 100] [--solvers bruteforce highs]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

from . import lexifair, reference_shim


# gym stand-ins at module level: GraphSubprocVecEnv pickles the spaces through its pipes (reference_shim's are local classes)
class _Env:
    def close(self):
        pass


class _Space:
    pass


class _Box(_Space):
    def __init__(self, low, high, shape=None, dtype=None):
        self.low, self.high, self.shape, self.dtype = low, high, shape, dtype


class _Discrete(_Space):
    def __init__(self, n):
        self.n = n


class _Tuple(_Space):
    def __init__(self, sp):
        self.spaces = sp


def _install_picklable_gym():
    mod = reference_shim._mod
    spaces = mod("gym.spaces", Box=_Box, Discrete=_Discrete, Tuple=_Tuple)
    reg = mod("gym.envs.registration", register=lambda **k: None)
    mod("gym", Env=_Env, Space=_Space, spaces=spaces, envs=mod("gym.envs", registration=reg), _fairmarl_stub=True)


def _solver(name):
    if name == "highs":
        return lambda costs: lexifair.lexifair_milp(np.asarray(costs, dtype=np.float64))
    return lexifair.solve_fair_assignment


def run(num_envs: int, num_agents: int, num_obstacles: int, steps: int, solver: str, fairness: bool = True):
    _install_picklable_gym()
    reference_shim.install_stubs(_solver(solver))           # registered in the parent before the fork (SURVEY 9.8)
    scen = "navigation_graph" if fairness else "nav_graph_goalassign_noFair"
    sys.argv = ["x"]
    from onpolicy.config import get_config
    parser = get_config()
    # the env arguments train_mpe.py adds (onpolicy/scripts/train_mpe.py parse_args)
    for flag, typ, default in (("--scenario_name", str, scen), ("--num_landmarks", int, num_agents), ("--num_agents", int, num_agents),
                               ("--num_obstacles", int, num_obstacles), ("--collaborative", bool, False), ("--max_speed", float, 2),
                               ("--collision_rew", float, 30), ("--goal_rew", float, 30), ("--min_dist_thresh", float, 0.05),
                               ("--use_dones", bool, False), ("--num_walls", int, 0), ("--zeroshift", float, 5), ("--fair_wt", float, 1),
                               ("--fair_rew", float, 1), ("--num_scripted_agents", int, 0), ("--world_size", float, 2),
                               ("--graph_feat_type", str, "relative"), ("--max_edge_dist", float, 1)):
        try:
            parser.add_argument(flag, type=typ, default=default)
        except argparse.ArgumentError:
            parser.set_defaults(**{flag[2:]: default})
    args = parser.parse_known_args([])[0]
    args.env_name, args.n_rollout_threads, args.episode_length, args.seed = "GraphMPE", num_envs, 25, 1
    args.scenario_name, args.num_agents, args.num_landmarks, args.num_obstacles = scen, num_agents, num_agents, num_obstacles
    # multiagent/custom_scenarios/__init__.py uses the removed `imp` module: provide `load` through importlib
    import importlib.util
    import types
    pkg = types.ModuleType("multiagent.custom_scenarios")
    pkg.__path__ = [os.path.join(reference_shim.REFERENCE_ROOT, "multiagent", "custom_scenarios")]

    def load(name):
        spec = importlib.util.spec_from_file_location("_ref_scn_" + name[:-3], os.path.join(pkg.__path__[0], name))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    pkg.load = load
    sys.modules["multiagent.custom_scenarios"] = pkg
    from multiagent.MPE_env import GraphMPEEnv
    from onpolicy.envs.env_wrappers import GraphSubprocVecEnv

    def get_env_fn(rank):
        def init_env():
            env = GraphMPEEnv(args)
            env.seed(args.seed + rank * 1000)
            return env
        return init_env
    envs = GraphSubprocVecEnv([get_env_fn(i) for i in range(num_envs)])
    envs.reset()
    rng = np.random.default_rng(0)
    eye = np.eye(5)
    warm = 5
    for k in range(warm):
        envs.step(eye[rng.integers(0, 5, (num_envs, num_agents))])
    t0 = time.perf_counter()
    for k in range(steps):
        obs, ag, node, adj, rew, done, infos = envs.step(eye[rng.integers(0, 5, (num_envs, num_agents))])
    dt = time.perf_counter() - t0
    envs.close()
    return {"impl": "reference GraphSubprocVecEnv (unmodified env, one process per env)", "solver_stub": solver,
            "num_envs": num_envs, "agents": num_agents, "obstacles": num_obstacles, "steps": steps, "seconds": dt,
            "agent_steps_per_s": num_envs * num_agents * steps / dt, "host_cores": os.cpu_count(),
            "obs_shape": list(obs.shape), "node_obs_shape": list(node.shape), "adj_shape": list(adj.shape)}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[os.cpu_count() or 1, 128])
    ap.add_argument("--agents", type=int, default=3)
    ap.add_argument("--obstacles", type=int, default=3)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--solvers", nargs="+", default=["bruteforce", "highs"])
    a = ap.parse_args()
    for s in a.solvers:
        for n in a.envs:
            print(json.dumps(run(n, a.agents, a.obstacles, a.steps, s)), flush=True)
