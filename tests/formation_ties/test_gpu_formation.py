"""The formation kernels' in-kernel lexifair solvers on exactly tied costs: lexifair_small<N> (csrc/fm_small.cuh) on the split
logic kernel and the fused kernel at N <= 4, lexifair_serial<N> (csrc/fm_form.cuh) on the fused kernel at N = 5 ... 7.  FA and
FA+FR re-solve the assignment on every step from the agent -> goal distances.  Positions reached by rollouts never tie, so
these states are built by hand: agents on a lattice of spacing 1 and goals on a 1/8 grid, in symmetric arrangements, so
that the distance matrix holds exact ties.  Velocities are zero, actions no-ops, obstacles and walls far away, and agents
at least 1 apart: the contact terms are below half an ulp of every coordinate, so the solve sees the positions as set.
Each case asserts that its costs tie and that the opposite tie rule (ties taken by descending (i, j)) would give a
different goal_match for some env, so a solver that broke ties the wrong way fails it."""
import numpy as np
import pytest

from oracle.formation import FormationConfig, FormationOracle, _norm
from oracle.lexifair import lexifair
from parity_util import assert_close
from test_gpu_formation import (_actions, _compare_step, _fp32, _from_device, _np, _sim, _to_device, _walls_from_device,
                                _walls_to_device)

pytestmark = pytest.mark.gpu

LATTICE = np.array([(x, y) for x in (-1.5, -0.5, 0.5, 1.5) for y in (-1.5, -0.5, 0.5, 1.5)])


def _costs(st):
    B, N = st.goal_match.shape
    return np.array([[[_norm(st.pos[b, a] - st.landmark_pos[b, g]) for g in range(N)] for a in range(N)] for b in range(B)])


def _reversed_tie_rule(costs):
    """The lexifair answer when tied entries are ordered by descending (i, j) instead: the same solver on the matrix with rows
    and columns reversed, mapped back."""
    n = costs.shape[-1]
    return n - 1 - lexifair(costs[:, ::-1, ::-1])[:, ::-1]


def _tied_state(cfg: FormationConfig, B: int, seed: int):
    N, O, W = cfg.num_agents, cfg.num_obstacles, cfg.num_walls
    rng = np.random.default_rng(seed)
    orc = FormationOracle(cfg, B, seed=seed)
    orc.reset()
    st = orc.get_state()
    for b in range(B):
        while True:                                                     # not every agent on a goal: no early reset
            agents = LATTICE[rng.choice(len(LATTICE), N, replace=False)]
            kind = b % 4
            if kind == 0:
                goals = -agents                                         # point reflection: cost[i][j] == cost[j][i]
            elif kind == 1:
                goals = np.stack([-agents[:, 1], agents[:, 0]], 1)      # quarter turn
            elif kind == 2:
                goals = rng.integers(-12, 13, (N, 2)) / 8               # 1/8 grid: 3-4-5 triangles and coincident goals
            else:
                goals = LATTICE[rng.integers(0, len(LATTICE), N)]       # lattice goals, some shared, some under an agent
            near = np.sqrt(((agents[:, None] - goals[None]) ** 2).sum(-1)).min(1) <= cfg.min_dist_thresh
            if not near.all():
                break
        st.pos[b], st.landmark_pos[b] = agents, goals
    st.obstacle_pos[:] = np.array([(6.0 + 2 * k, 6.0) for k in range(O)]).reshape(1, O, 2)
    st.vel[:] = 0.0
    st.goal_match[:] = np.arange(N)
    st.status[:] = False
    st.step[:] = 0
    st.goal_reached[:] = -1.0
    st.goal_history[:] = -1.0
    st.occupied[:] = 0.0
    if W:
        orc.wall_axis[:] = np.array([6.0, -6.0])[:W]
        orc.wall_orient[:] = np.array([0, 1])[:W]
        orc.wall_len[:] = 0.5
    st = _fp32(st)
    orc.set_state(st)
    return st, orc


def _case(N, O, W, fused, fair):
    return pytest.param(N, O, W, fused, fair, id=f"{N}-{O}-{W}-{'fused' if fused else 'split' if N <= 4 and O <= 3 and not W else 'fused_only'}-{'fafr' if fair else 'fa'}")


TIE_CASES = [
    _case(2, 1, 0, False, True), _case(3, 2, 0, False, False), _case(4, 3, 0, False, True),      # split logic kernel: lexifair_small
    _case(2, 0, 0, True, False), _case(3, 1, 0, True, True), _case(4, 2, 0, True, False),        # fused kernel: lexifair_small
    _case(5, 1, 0, False, True), _case(6, 2, 0, False, False), _case(7, 3, 0, False, True),      # fused kernel: lexifair_serial
    _case(4, 1, 2, False, True),                                                                 # two walls (fused kernel)
]


@pytest.mark.parametrize("N,O,W,fused,fair", TIE_CASES)
def test_tied_costs_match_oracle_for_one_and_three_steps(N, O, W, fused, fair, monkeypatch):
    import fair_marl_b200 as fm
    if fused:
        monkeypatch.setenv("FM_FORM_FUSED", "1")
    B = 64
    cfg = FormationConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=25,
                          fairness_reward=fair, assignment="fair", num_walls=W)
    st, orc = _tied_state(cfg, B, seed=10 * N + O + W)
    costs = _costs(st)
    want = lexifair(costs)
    tied = [np.unique(c).size < c.size for c in costs]
    assert sum(tied) >= B // 2
    assert (want != _reversed_tie_rule(costs)).any(1).sum() >= 1, "no env where the tie rule decides the assignment"
    env = fm.B200FormationVecEnv(_sim(cfg), num_envs=B, seed=3)
    env.set_state({**_to_device(st), **_walls_to_device(orc)})
    a = np.zeros((B, N), np.int64)
    for t in range(3):
        dev = env.get_state()
        cur = _from_device(dev)
        orc.set_state(cur)
        _walls_from_device(orc, dev)
        out = _np(env.step_tensor(_actions(a)))
        ref = orc.step(a, autoreset=True)
        post, rpost = _from_device(env.get_state()), orc.get_state()
        assert not ref["reset"].any()
        assert (post.pos == st.pos).all() and (rpost.pos == st.pos).all(), "an agent moved: the costs are not the set ones"
        _compare_step(out, ref, post, rpost)                                 # goal_match bit for bit
        assert (post.goal_match == want).all(), t
        for f in ("vel", "p_dist", "dists_to_goal", "times_required", "dist_left_to_goal", "occupied", "goal_history",
                  "goal_reached", "min_time"):
            assert_close(getattr(post, f), getattr(rpost, f), f)
    env.close()
