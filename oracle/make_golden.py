"""Generate tests/golden/*.npz by running the UNMODIFIED reference (TEST INFRASTRUCTURE ONLY).

Run with FAIRMARL_REFERENCE_ROOT set to a checkout of the original project:

    FAIRMARL_REFERENCE_ROOT=<checkout> python -m oracle.make_golden

For every config a single reference ``MultiAgentGraphEnv`` (built exactly as
multiagent/MPE_env.py:62-75 builds it, with the two stubs of
oracle/reference_shim.py) is rolled for a few episodes.  Half of the episodes use
goal-seeking actions so goal latches, agent collisions and obstacle collisions
fire.  Per step we record the pre-step state, the action indices, every output
of ``env.step`` (obs, node_obs, adj, reward, done, the 14 info keys) and the
post-step state; per reset the outputs of ``env.reset`` and the post-reset state.
All values are float64 exactly as the reference produced them.
"""
from __future__ import annotations

import os
from dataclasses import asdict, fields

import numpy as np

from .navgraph import INFO_KEYS, NavConfig, NavState
from .reference_shim import extract_state, make_reference_env

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

CONFIGS = {
    # name: (config, reference seed, episodes)
    "n3_o3_fafr": (NavConfig(num_agents=3, num_obstacles=3, goal_rew=30.0, collision_rew=30.0), 11, 8),
    "n3_o3_fa": (NavConfig(num_agents=3, num_obstacles=3, fairness_reward=False), 12, 6),
    "n7_o3_fafr": (NavConfig(num_agents=7, num_obstacles=3), 13, 4),
    "n5_o0_fafr": (NavConfig(num_agents=5, num_obstacles=0), 14, 4),
    "n16_o3_fafr": (NavConfig(num_agents=16, num_obstacles=3), 15, 2),
    "n4_o2_collab": (NavConfig(num_agents=4, num_obstacles=2, collaborative=True), 16, 3),
    "n3_o3_global": (NavConfig(num_agents=3, num_obstacles=3, graph_feat_type="global"), 17, 4),
    "n7_o3_global": (NavConfig(num_agents=7, num_obstacles=3, graph_feat_type="global"), 18, 2),
    # walls (oracle and the wall instantiations of the group-per-env kernels)
    "n3_o3_w2": (NavConfig(num_agents=3, num_obstacles=3, num_walls=2), 19, 12),
    "n4_o2_w1": (NavConfig(num_agents=4, num_obstacles=2, num_walls=1, goal_rew=30.0, collision_rew=30.0), 20, 9),
}


def _seek_actions(state: NavState, rng, p_random: float) -> np.ndarray:
    """Greedy move towards the assigned goal (action meaning: environment.py:301-311 ->
    0 no-op, 1 +x, 2 -x, 3 +y, 4 -y), with probability p_random a uniform action instead."""
    goal = state.landmark_pos[0][state.goal_match[0]]
    d = goal - state.pos[0]
    a = np.where(np.abs(d[:, 0]) > np.abs(d[:, 1]), np.where(d[:, 0] > 0, 1, 2), np.where(d[:, 1] > 0, 3, 4))
    rnd = rng.random(a.shape[0]) < p_random
    return np.where(rnd, rng.integers(0, 5, a.shape[0]), a)


def _seek_walls(state: NavState, rng, p_random: float) -> np.ndarray:
    """Drive every agent at the nearest point of wall (agent index mod W), ends included, so that the fixtures hold
    wall contact forces in both branches of core.py:417-432 and wall-box collisions (navigation_graph.py:670-683)."""
    N, W = state.pos.shape[1], state.wall_axis.shape[1]
    a = np.zeros(N, dtype=np.int64)
    for i in range(N):
        w = i % W
        horiz = state.wall_orient[0, w] == 0
        L = state.wall_len[0]
        along = np.clip(state.pos[0, i, 0 if horiz else 1], -1.3 * L, 1.3 * L)   # aim slightly past the ends too
        target = np.array([along, state.wall_axis[0, w]]) if horiz else np.array([state.wall_axis[0, w], along])
        d = target - state.pos[0, i]
        a[i] = (1 if d[0] > 0 else 2) if abs(d[0]) > abs(d[1]) else (3 if d[1] > 0 else 4)
    rnd = rng.random(N) < p_random
    return np.where(rnd, rng.integers(0, 5, N), a)


def _stack_states(states):
    return {"state_" + f.name: np.concatenate([getattr(s, f.name) for s in states], axis=0)
            for f in fields(NavState) if getattr(states[0], f.name) is not None}


def generate(name: str) -> str:
    cfg, seed, episodes = CONFIGS[name]
    env, sc = make_reference_env(cfg, seed=seed)
    rng = np.random.default_rng(seed)
    N = cfg.num_agents
    pre, post, acts = [], [], []
    outs = {k: [] for k in ("obs", "node_obs", "adj", "reward", "done")}
    infos = {k: [] for k in INFO_KEYS}
    r_state, r_obs, r_node, r_adj, r_prev_match = [], [], [], [], []
    for ep in range(episodes):
        prev_match = np.array(sc.goal_match_index).copy()
        o = env.reset()
        st = extract_state(env, sc)
        r_state.append(st)
        r_prev_match.append(prev_match[None])
        r_obs.append(np.array(o[0])[None])
        r_node.append(np.array(o[2])[None])
        r_adj.append(np.array(o[3])[0][None])
        for t in range(cfg.episode_length):
            st = extract_state(env, sc)
            if cfg.num_walls and ep % 3 == 2:
                a = _seek_walls(st, rng, 0.2)
            else:
                a = rng.integers(0, 5, N) if ep % 2 == 0 else _seek_actions(st, rng, 0.15)
            oh = np.eye(5)[a]
            ob, ag_id, node, adj, rew, done, info = env.step([oh[i] for i in range(N)])
            pre.append(st)
            acts.append(a[None])
            post.append(extract_state(env, sc))
            outs["obs"].append(np.array(ob)[None])
            outs["node_obs"].append(np.array(node)[None])
            outs["adj"].append(np.array(adj)[0][None])
            outs["reward"].append(np.array(rew, dtype=np.float64).reshape(1, N))
            outs["done"].append(np.array(done)[None])
            for k in INFO_KEYS:
                infos[k].append(np.array([[info[i][k] for i in range(N)]], dtype=np.float64))
    data = {"config_" + k: np.array(v) for k, v in asdict(cfg).items()}
    data.update({"pre_" + k[6:]: v for k, v in _stack_states(pre).items()})
    data.update({"post_" + k[6:]: v for k, v in _stack_states(post).items()})
    data.update({"reset_" + k[6:]: v for k, v in _stack_states(r_state).items()})
    data["reset_prev_goal_match"] = np.concatenate(r_prev_match)
    data["reset_obs"] = np.concatenate(r_obs)
    data["reset_node_obs"] = np.concatenate(r_node)
    data["reset_adj"] = np.concatenate(r_adj)
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
    """-> (NavConfig, dict of arrays)."""
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    kw = {}
    for f in fields(NavConfig):
        if "config_" + f.name in z.files:            # fixtures written before a field existed keep its default
            kw[f.name] = z["config_" + f.name].item()
    cfg = NavConfig(**kw)
    return cfg, {k: z[k] for k in z.files if not k.startswith("config_")}


def state_from(data, prefix: str, sl=slice(None)) -> NavState:
    # optional fields (walls) are absent from fixtures of configs without them
    return NavState(**{f.name: (data[prefix + f.name][sl] if prefix + f.name in data else None) for f in fields(NavState)})


if __name__ == "__main__":
    import sys
    for n in (sys.argv[1:] or CONFIGS):
        p = generate(n)
        print(n, "->", p, os.path.getsize(p) // 1024, "KiB")
