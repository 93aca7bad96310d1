"""Import the UNMODIFIED reference env as a checker (TEST INFRASTRUCTURE ONLY).

Only usable where ``FAIRMARL_REFERENCE_ROOT`` names a checkout of the original Fair-MARL
project, which this repository does not contain; nothing in ``-m gpu`` tests / smoke / bench imports this.
Recipe: SURVEY.md Appendix A -- stub ``gym`` (absent) and ``marl_fair_assign``
(needs pyomo + gurobi) in ``sys.modules``, load the scenario file by path
(``custom_scenarios/__init__.py`` uses the removed ``imp`` module), and wire the
callbacks exactly as ``multiagent/MPE_env.py:62-75`` does.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types
from argparse import Namespace

import numpy as np

from . import lexifair
from .navgraph import NavConfig, NavState

REFERENCE_ROOT = os.environ.get("FAIRMARL_REFERENCE_ROOT", "")
SKIP_REASON = "needs the original Fair-MARL project: set FAIRMARL_REFERENCE_ROOT to its checkout"


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "multiagent", "core.py"))


def _mod(name, **kw):
    m = types.ModuleType(name)
    m.__dict__.update(kw)
    m.__path__ = []
    sys.modules[name] = m
    return m


def install_stubs(solver=lexifair.solve_fair_assignment) -> None:
    if "gym" not in sys.modules or not hasattr(sys.modules["gym"], "_fairmarl_stub"):
        class Env:
            def close(self):
                pass

        class Space:
            pass

        class Box(Space):
            def __init__(self, low, high, shape=None, dtype=None):
                self.low, self.high, self.shape, self.dtype = low, high, shape, dtype

        class Discrete(Space):
            def __init__(self, n):
                self.n = n

        class Tuple(Space):
            def __init__(self, sp):
                self.spaces = sp

        spaces = _mod("gym.spaces", Box=Box, Discrete=Discrete, Tuple=Tuple)
        reg = _mod("gym.envs.registration", register=lambda **k: None)
        _mod("gym", Env=Env, Space=Space, spaces=spaces, envs=_mod("gym.envs", registration=reg),
             _fairmarl_stub=True)
    _mod("marl_fair_assign", solve_fair_assignment=solver)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


def args_from_config(cfg: NavConfig) -> Namespace:
    return Namespace(
        num_agents=cfg.num_agents, num_landmarks=cfg.num_agents, world_size=cfg.world_size,
        num_scripted_agents=0, num_obstacles=cfg.num_obstacles, collaborative=cfg.collaborative,
        max_speed=cfg.max_speed, collision_rew=cfg.collision_rew, goal_rew=cfg.goal_rew,
        min_dist_thresh=cfg.min_dist_thresh, use_dones=False, episode_length=cfg.episode_length,
        max_edge_dist=cfg.max_edge_dist, graph_feat_type=cfg.graph_feat_type, fair_wt=1, fair_rew=cfg.fair_rew,
        num_walls=cfg.num_walls, zeroshift=cfg.zeroshift, scenario_name="navigation_graph",
        algorithm_name="rmappo")


def _load_scenario(file_name: str):
    path = os.path.join(REFERENCE_ROOT, "multiagent", "custom_scenarios", file_name)
    spec = importlib.util.spec_from_file_location("_fairmarl_ref_" + file_name[:-3], path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def make_reference_env(cfg: NavConfig, seed: int = 0):
    """Reference ``GraphMPEEnv(args)`` (MPE_env.py:55-77) for ``cfg``.  Returns (env, scenario)."""
    install_stubs()
    fname = "navigation_graph.py" if cfg.fairness_reward else "nav_graph_goalassign_noFair.py"
    nav = _load_scenario(fname)
    from multiagent.environment import MultiAgentGraphEnv
    np.random.seed(seed)
    scenario = nav.Scenario()
    world = scenario.make_world(args=args_from_config(cfg))
    env = MultiAgentGraphEnv(
        world=world, reset_callback=scenario.reset_world, reward_callback=scenario.reward,
        observation_callback=scenario.observation, graph_observation_callback=scenario.graph_observation,
        update_graph=scenario.update_graph, id_callback=scenario.get_id,
        info_callback=scenario.info_callback, done_callback=scenario.done,
        scenario_name="navigation_graph")
    env.seed(seed)
    return env, scenario


def extract_state(env, scenario) -> NavState:
    """Single-env NavState (B = 1) from the live reference objects."""
    w = env.world
    N = len(w.agents)
    return NavState(
        pos=np.array([[a.state.p_pos for a in w.agents]], dtype=np.float64),
        vel=np.array([[a.state.p_vel for a in w.agents]], dtype=np.float64),
        p_dist=np.array([[a.state.p_dist for a in w.agents]], dtype=np.float64),
        landmark_pos=np.array([[l.state.p_pos for l in w.landmarks]], dtype=np.float64),
        obstacle_pos=np.array([[o.state.p_pos for o in w.obstacles]], dtype=np.float64).reshape(1, len(w.obstacles), 2),
        goal_match=np.array([scenario.goal_match_index], dtype=np.int64),
        dists_to_goal=np.array([w.dists_to_goal], dtype=np.float64),
        times_required=np.array([w.times_required], dtype=np.float64),
        dist_left_to_goal=np.array([w.dist_left_to_goal], dtype=np.float64),
        num_agent_collisions=np.array([w.num_agent_collisions], dtype=np.float64),
        num_obstacle_collisions=np.array([w.num_obstacle_collisions], dtype=np.float64),
        dist_traveled_mean=np.array([getattr(w, "dist_traveled_mean", 0.0)], dtype=np.float64),
        dist_traveled_stddev=np.array([getattr(w, "dist_traveled_stddev", 0.0)], dtype=np.float64),
        step=np.array([env.current_step], dtype=np.int64),
        min_time=np.array([[a.goal_min_time for a in w.agents]], dtype=np.float64),
        episode=np.zeros(1, dtype=np.int64),
        wall_axis=np.array([[wl.axis_pos for wl in w.walls]], dtype=np.float64) if len(w.walls) else None,
        wall_orient=np.array([[0 if wl.orient == "H" else 1 for wl in w.walls]], dtype=np.int64) if len(w.walls) else None,
        wall_len=np.array([scenario.wall_length], dtype=np.float64) if len(w.walls) else None)


def inject_state(env, scenario, st: NavState, b: int = 0) -> None:
    """Write env ``b`` of ``st`` into the live reference objects (SURVEY.md section 8c recipe)."""
    w = env.world
    for i, a in enumerate(w.agents):
        a.state.p_pos = np.array(st.pos[b, i], dtype=np.float64)
        a.state.p_vel = np.array(st.vel[b, i], dtype=np.float64)
        a.state.p_dist = float(st.p_dist[b, i])
        a.goal_min_time = float(st.min_time[b, i])
    for i, l in enumerate(w.landmarks):
        l.state.p_pos = np.array(st.landmark_pos[b, i], dtype=np.float64)
        l.state.p_vel = np.zeros(2)
    for i, o in enumerate(w.obstacles):
        o.state.p_pos = np.array(st.obstacle_pos[b, i], dtype=np.float64)
        o.state.p_vel = np.zeros(2)
    for i, wl in enumerate(w.walls):                  # what random_scenario sets per episode (navigation_graph.py:294-324)
        scenario.wall_length = float(st.wall_len[b])
        wl.orient = "H" if int(st.wall_orient[b, i]) == 0 else "V"
        wl.width, wl.hard = 0.1, True
        wl.endpoints = np.array([-scenario.wall_length, scenario.wall_length])
        wl.axis_pos = float(st.wall_axis[b, i])
        wl.state.p_pos = np.array([0.0, wl.axis_pos]) if wl.orient == "H" else np.array([wl.axis_pos, 0.0])
        wl.state.p_vel = np.zeros(2)
    scenario.goal_match_index = np.array(st.goal_match[b], dtype=np.int64)
    w.dists_to_goal = np.array(st.dists_to_goal[b], dtype=np.float64)
    w.times_required = np.array(st.times_required[b], dtype=np.float64)
    w.dist_left_to_goal = np.array(st.dist_left_to_goal[b], dtype=np.float64)
    w.num_agent_collisions = np.array(st.num_agent_collisions[b], dtype=np.float64)
    w.num_obstacle_collisions = np.array(st.num_obstacle_collisions[b], dtype=np.float64)
    w.dist_traveled_mean = float(st.dist_traveled_mean[b])
    w.dist_traveled_stddev = float(st.dist_traveled_stddev[b])
    env.current_step = int(st.step[b])
    w.current_time_step = int(st.step[b])
    for a in w.agents:
        a.state.time = 0.0
        for _ in range(int(st.step[b])):
            a.state.time += w.dt
    w.calculate_distances()
