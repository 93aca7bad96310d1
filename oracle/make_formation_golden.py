"""Record formation-family fixtures from the UNMODIFIED reference (needs FAIRMARL_REFERENCE_ROOT; TEST INFRASTRUCTURE).

    python -m oracle.make_formation_golden            # writes tests/golden/formation_*.npz

Each fixture holds, per recorded step of the live reference env (``MultiAgentGraphEnv`` over
``nav_fairassign_fairrew_formation_graph.Scenario`` / its ``nofairrew`` twin / the base scenarios
``nav_base_formation_graph_mask`` and ``..._randomgoal``): the full pre-step state, the actions,
the 7-tuple outputs and info dicts, and the post-step state; plus the post-reset states and reset outputs.  Half of
the episodes steer the agents at their assigned goals (with noise) so that ``agent.status`` latches, goals get
occupied / vacated and the early ``done`` path is taken; the rest are random walks.
"""
from __future__ import annotations

import os
from dataclasses import asdict, fields

import numpy as np

from .formation import FormationConfig, FormationState
from .navgraph import INFO_KEYS
from .reference_shim import _load_scenario, args_from_config, install_stubs

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# name -> (config, seed, episodes)
CONFIGS = {
    "formation_n3_o3_fafr": (FormationConfig(num_agents=3, num_obstacles=3, goal_rew=30.0, collision_rew=30.0), 31, 14),
    "formation_n4_o2_fa": (FormationConfig(num_agents=4, num_obstacles=2, fairness_reward=False, min_obs_dist=0.8,
                                           episode_length=20), 32, 12),
    "formation_n7_o3_fafr": (FormationConfig(num_agents=7, num_obstacles=3, collaborative=True, episode_length=30), 33, 8),
    # the base formation scenarios of model_weights/OA and RA (config.yaml: 3 agents, 3 obstacles, rewards 30)
    "formation_n3_o3_oa": (FormationConfig(num_agents=3, num_obstacles=3, goal_rew=30.0, collision_rew=30.0,
                                           fairness_reward=False, assignment="optimal"), 34, 10),
    "formation_n3_o3_ra": (FormationConfig(num_agents=3, num_obstacles=3, goal_rew=30.0, collision_rew=30.0,
                                           fairness_reward=False, assignment="random"), 35, 10),
    # walls in this family (box test 1.5 * size, wall.id in the node rows, wall length redrawn per reset)
    "formation_n3_o2_w2": (FormationConfig(num_agents=3, num_obstacles=2, num_walls=2, goal_rew=30.0, collision_rew=30.0), 36, 12),
    "formation_n3_o3_w1_oa": (FormationConfig(num_agents=3, num_obstacles=3, num_walls=1, goal_rew=30.0, collision_rew=30.0,
                                              fairness_reward=False, assignment="optimal"), 37, 9),
}

SCENARIO_FILES = {("fair", True): "nav_fairassign_fairrew_formation_graph.py",
                  ("fair", False): "nav_fairassign_nofairrew_formation_graph.py",
                  ("optimal", False): "nav_base_formation_graph_mask.py",
                  ("random", False): "nav_base_formation_graph_randomgoal.py"}


def make_reference_env(cfg: FormationConfig, seed: int):
    install_stubs()
    mod = _load_scenario(SCENARIO_FILES[(cfg.assignment, bool(cfg.fairness_reward))])
    from multiagent.environment import MultiAgentGraphEnv
    np.random.seed(seed)
    sc = mod.Scenario()
    args = args_from_config(cfg)
    args.min_obs_dist = cfg.min_obs_dist
    world = sc.make_world(args=args)
    env = MultiAgentGraphEnv(
        world=world, reset_callback=sc.reset_world, reward_callback=sc.reward, observation_callback=sc.observation,
        graph_observation_callback=sc.graph_observation, update_graph=sc.update_graph, id_callback=sc.get_id,
        info_callback=sc.info_callback, done_callback=sc.done, scenario_name="nav_fairassign_fairrew_formation_graph")
    env.seed(seed)
    return env, sc


def extract_state(env, sc) -> FormationState:
    w = env.world
    f64 = lambda x: np.array([x], dtype=np.float64)
    return FormationState(
        pos=f64([a.state.p_pos for a in w.agents]), vel=f64([a.state.p_vel for a in w.agents]),
        p_dist=f64([a.state.p_dist for a in w.agents]), landmark_pos=f64(sc.landmark_poses),
        obstacle_pos=f64([o.state.p_pos for o in w.obstacles]).reshape(1, len(w.obstacles), 2),
        # the mask scenario calls it optimal_match_index (set at reset only)
        goal_match=np.array([sc.goal_match_index if hasattr(sc, "goal_match_index") else sc.optimal_match_index],
                            dtype=np.int64), dists_to_goal=f64(w.dists_to_goal),
        times_required=f64(w.times_required), dist_left_to_goal=f64(w.dist_left_to_goal),
        num_agent_collisions=f64(w.num_agent_collisions), num_obstacle_collisions=f64(w.num_obstacle_collisions),
        dist_traveled_mean=f64(getattr(w, "dist_traveled_mean", 0.0)),
        dist_traveled_stddev=f64(getattr(w, "dist_traveled_stddev", 0.0)),
        step=np.array([env.current_step], dtype=np.int64), min_time=f64([a.goal_min_time for a in w.agents]),
        episode=np.zeros(1, dtype=np.int64), status=np.array([[a.status is True for a in w.agents]]),
        goal_reached=f64(sc.goal_reached), occupied=f64(sc.landmark_poses_occupied), goal_history=f64(sc.goal_history))


def extract_walls(env, sc):
    """(wall_axis [1,W], wall_orient [1,W] (0 = 'H', 1 = 'V'), wall_len [1]) of the live reference."""
    w = env.world.walls
    return (np.array([[x.axis_pos for x in w]], dtype=np.float64).reshape(1, len(w)),
            np.array([[0 if x.orient == "H" else 1 for x in w]], dtype=np.int64).reshape(1, len(w)),
            np.array([sc.wall_length], dtype=np.float64))


def _seek_walls(st: FormationState, walls, rng, p_random: float) -> np.ndarray:
    """Drive every agent at the nearest point of wall (agent index mod W), slightly past its ends too."""
    axis, orient, length = walls
    N, W = st.pos.shape[1], axis.shape[1]
    a = np.zeros(N, dtype=np.int64)
    for i in range(N):
        w = i % W
        horiz = orient[0, w] == 0
        along = np.clip(st.pos[0, i, 0 if horiz else 1], -1.3 * length[0], 1.3 * length[0])
        target = np.array([along, axis[0, w]]) if horiz else np.array([axis[0, w], along])
        d = target - st.pos[0, i]
        a[i] = (1 if d[0] > 0 else 2) if abs(d[0]) > abs(d[1]) else (3 if d[1] > 0 else 4)
    return np.where(rng.random(N) < p_random, rng.integers(0, 5, N), a)


def _seek(st: FormationState, rng, p_random: float) -> np.ndarray:
    """Greedy axis move towards the assigned goal, random with probability p_random."""
    N = st.pos.shape[1]
    a = np.zeros(N, dtype=np.int64)
    for i in range(N):
        d = st.landmark_pos[0, st.goal_match[0, i]] - st.pos[0, i]
        a[i] = (1 if d[0] > 0 else 2) if abs(d[0]) > abs(d[1]) else (3 if d[1] > 0 else 4)
    return np.where(rng.random(N) < p_random, rng.integers(0, 5, N), a)


def _stack(states, prefix):
    return {prefix + f.name: np.concatenate([getattr(s, f.name) for s in states], axis=0) for f in fields(FormationState)}


def generate(name: str) -> str:
    cfg, seed, episodes = CONFIGS[name]
    env, sc = make_reference_env(cfg, seed)
    rng = np.random.default_rng(seed)
    N = cfg.num_agents
    pre, post, acts, resets = [], [], [], []
    outs = {k: [] for k in ("obs", "node_obs", "adj", "reward", "done")}
    infos = {k: [] for k in INFO_KEYS}
    r_obs, r_node, r_adj = [], [], []
    walls_pre, walls_reset = [], []
    for ep in range(episodes):
        o = env.reset()
        resets.append(extract_state(env, sc))
        walls_reset.append(extract_walls(env, sc))
        r_obs.append(np.array(o[0])[None]); r_node.append(np.array(o[2])[None]); r_adj.append(np.array(o[3])[0][None])
        for t in range(cfg.episode_length):
            st = extract_state(env, sc)
            if cfg.num_walls and ep % 3 == 2:
                a = _seek_walls(st, extract_walls(env, sc), rng, 0.2)
            else:
                a = rng.integers(0, 5, N) if ep % 2 else _seek(st, rng, 0.1 if ep % 4 == 0 else 0.3)
            walls_pre.append(extract_walls(env, sc))
            oh = np.eye(5)[a]
            ob, ag_id, node, adj, rew, done, info = env.step([oh[i] for i in range(N)])
            pre.append(st); acts.append(a[None]); post.append(extract_state(env, sc))
            outs["obs"].append(np.array(ob)[None]); outs["node_obs"].append(np.array(node)[None])
            outs["adj"].append(np.array(adj)[0][None])
            outs["reward"].append(np.array(rew, dtype=np.float64).reshape(1, N))
            outs["done"].append(np.array(done)[None])
            for k in INFO_KEYS:
                infos[k].append(np.array([[info[i][k] for i in range(N)]], dtype=np.float64))
            if all(done):                                  # graphworker would reset here (env_wrappers.py:859-865)
                break
    data = {"config_" + k: np.array(v) for k, v in asdict(cfg).items()}
    data.update(_stack(pre, "pre_")); data.update(_stack(post, "post_")); data.update(_stack(resets, "reset_"))
    data["reset_obs"], data["reset_node_obs"], data["reset_adj"] = map(np.concatenate, (r_obs, r_node, r_adj))
    if cfg.num_walls:
        for prefix, rec in (("pre_", walls_pre), ("reset_", walls_reset)):
            for k, field in enumerate(("wall_axis", "wall_orient", "wall_len")):
                data[prefix + field] = np.concatenate([r[k] for r in rec], axis=0)
    data["actions"] = np.concatenate(acts)
    for k, v in outs.items():
        data["out_" + k] = np.concatenate(v)
    for k, v in infos.items():
        data["info_" + k] = np.concatenate(v)
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    path = os.path.join(GOLDEN_DIR, name + ".npz")
    np.savez_compressed(path, **data)
    return path


def load(name: str):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    kw = {f.name: z["config_" + f.name].item() for f in fields(FormationConfig) if "config_" + f.name in z.files}
    return FormationConfig(**kw), {k: z[k] for k in z.files if not k.startswith("config_")}


def set_walls(orc, data, prefix: str) -> None:
    """Load the recorded wall geometry (kept beside FormationState) into a FormationOracle."""
    if prefix + "wall_axis" in data:
        orc.wall_axis = data[prefix + "wall_axis"].astype(np.float64).copy()
        orc.wall_orient = data[prefix + "wall_orient"].astype(np.int64).copy()
        orc.wall_len = data[prefix + "wall_len"].astype(np.float64).copy()


def state_from(data, prefix: str) -> FormationState:
    return FormationState(**{f.name: data[prefix + f.name] for f in fields(FormationState)})


if __name__ == "__main__":
    import sys
    for n in (sys.argv[1:] or CONFIGS):
        p = generate(n)
        z = np.load(p)
        print(n, "->", p, os.path.getsize(p) // 1024, "KiB;", z["actions"].shape[0], "steps,",
              int(z["post_status"].any(axis=1).sum()), "with a latched agent,", int((z["pre_occupied"] == 1).any(axis=1).sum()),
              "with an occupied goal")


def inject_state(env, sc, st: FormationState, b: int = 0) -> None:
    """Write env ``b`` of ``st`` into the live reference objects (what reset_world / random_scenario / the callbacks set)."""
    w = env.world
    for i, a in enumerate(w.agents):
        a.state.p_pos = np.array(st.pos[b, i], dtype=np.float64)
        a.state.p_vel = np.array(st.vel[b, i], dtype=np.float64)
        a.state.p_dist = float(st.p_dist[b, i])
        a.goal_min_time = float(st.min_time[b, i])
        a.status = bool(st.status[b, i])
    for i, l in enumerate(w.landmarks):
        l.state.p_pos = np.array(st.landmark_pos[b, i], dtype=np.float64)
    for i, o in enumerate(w.obstacles):
        o.state.p_pos = np.array(st.obstacle_pos[b, i], dtype=np.float64)
    sc.landmark_poses = np.array(st.landmark_pos[b], dtype=np.float64)
    if hasattr(sc, "goal_match_index"):
        sc.goal_match_index = np.array(st.goal_match[b], dtype=np.int64)
    else:
        sc.optimal_match_index = np.array(st.goal_match[b], dtype=np.int64)
    sc.goal_reached = np.array(st.goal_reached[b], dtype=np.float64)
    sc.landmark_poses_occupied = np.array(st.occupied[b], dtype=np.float64)
    sc.goal_history = np.array(st.goal_history[b], dtype=np.float64)
    w.dists_to_goal = np.array(st.dists_to_goal[b], dtype=np.float64)
    w.times_required = np.array(st.times_required[b], dtype=np.float64)
    w.dist_left_to_goal = np.array(st.dist_left_to_goal[b], dtype=np.float64)
    w.num_agent_collisions = np.array(st.num_agent_collisions[b], dtype=np.float64)
    w.num_obstacle_collisions = np.array(st.num_obstacle_collisions[b], dtype=np.float64)
    w.dist_traveled_mean = float(st.dist_traveled_mean[b])
    w.dist_traveled_stddev = float(st.dist_traveled_stddev[b])
    env.current_step = int(st.step[b])
    w.current_time_step = int(st.step[b])
    w.calculate_distances()
