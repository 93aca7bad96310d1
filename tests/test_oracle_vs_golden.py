"""Pin the numpy oracle against golden vectors produced by the UNMODIFIED reference
(oracle/make_golden.py, run against a checkout of it)."""
import numpy as np
import pytest

from oracle.lexifair import lexifair
from oracle.make_golden import CONFIGS, load, state_from
from oracle.navgraph import INFO_KEYS, NavGraphOracle, NavState

TOL = 1e-11      # float64 restatement vs float64 reference: |a-b| <= TOL * max(1, |ref|)


def _close(a, b, tol=TOL):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    fin = np.isfinite(b)
    assert (np.isfinite(a) == fin).all()
    err = np.abs(a[fin] - b[fin]) / np.maximum(1.0, np.abs(b[fin]))
    assert err.size == 0 or err.max() <= tol, err.max()


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_step_matches_reference(name):
    cfg, g = load(name)
    T = g["actions"].shape[0]
    orc = NavGraphOracle(cfg, T)
    orc.set_state(state_from(g, "pre_"))
    out = orc.step(actions=g["actions"], autoreset=False)
    for k in ("obs", "node_obs", "adj", "reward"):
        _close(out[k], g["out_" + k])
    assert (out["done"] == g["out_done"]).all()
    for k in INFO_KEYS:
        _close(out["info"][k], g["info_" + k])
    post = orc.get_state()
    ref_post = state_from(g, "post_")
    for f in ("pos", "vel", "p_dist", "dists_to_goal", "times_required", "dist_left_to_goal",
              "num_agent_collisions", "num_obstacle_collisions", "dist_traveled_mean",
              "dist_traveled_stddev"):
        _close(getattr(post, f), getattr(ref_post, f))
    assert (post.step == ref_post.step).all()
    # the goldens exercise the interesting branches
    assert (g["info_Time_req_to_goal"] > 0).any(), "no goal latch in golden"
    assert (g["info_Num_agent_collisions"] > 0).any() or cfg.num_agents < 3


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_reset_outputs_and_assignment_match_reference(name):
    cfg, g = load(name)
    st = state_from(g, "reset_")
    R = st.pos.shape[0]
    orc = NavGraphOracle(cfg, R)
    orc.set_state(st)
    ob = orc.observe()
    _close(ob["obs"], g["reset_obs"])
    _close(ob["node_obs"], g["reset_node_obs"])
    _close(ob["adj"], g["reset_adj"])
    # navigation_graph.py:555-558: lexifair on cdist(agent_pos, goal_pos)
    d = st.pos[:, :, None, :] - st.landmark_pos[:, None, :, :]
    costs = np.sqrt(d[..., 0] ** 2 + d[..., 1] ** 2)
    assert (lexifair(costs) == st.goal_match).all()
    # navigation_graph.py:545-547: min_time uses the PREVIOUS episode's goal_match_index
    prev = g["reset_prev_goal_match"]
    old_goal = np.take_along_axis(st.landmark_pos, prev[..., None], axis=1)
    dd = st.pos - old_goal
    _close(st.min_time, np.sqrt(dd[..., 0] ** 2 + dd[..., 1] ** 2) / cfg.max_speed)
    # reset rules (a-14): zeroed metrics, zero velocity
    assert (st.vel == 0).all() and (st.p_dist == 0).all() and (st.step == 0).all()
    assert (st.dists_to_goal == -1).all() and (st.times_required == -1).all()


@pytest.mark.reference
def test_oracle_tracks_live_reference_rollout():
    """Roll the live reference and the oracle side by side (no state re-injection inside an episode)."""
    from oracle.navgraph import NavConfig
    from oracle.reference_shim import extract_state, make_reference_env
    cfg = NavConfig(num_agents=4, num_obstacles=3)
    env, sc = make_reference_env(cfg, seed=5)
    rng = np.random.default_rng(5)
    orc = NavGraphOracle(cfg, 1)
    for ep in range(3):
        env.reset()
        orc.set_state(extract_state(env, sc))
        for t in range(cfg.episode_length):
            a = rng.integers(0, 5, cfg.num_agents)
            oh = np.eye(5)[a]
            r = env.step([oh[i] for i in range(cfg.num_agents)])
            out = orc.step(actions=a[None], autoreset=False)
            _close(out["obs"][0], np.array(r[0]), 1e-9)
            _close(out["node_obs"][0], np.array(r[2]), 1e-9)
            _close(out["adj"][0], np.array(r[3])[0], 1e-9)
            _close(out["reward"][0], np.array(r[4], dtype=float).reshape(-1), 1e-9)
