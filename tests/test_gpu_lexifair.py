"""The stand-alone lexifair entries (fm_assign_costs / fm_assign_positions: assign_kernel<G> around lexifair_group<G>,
csrc/fm_kernels.cu and fm_device.cuh) against exact oracles, at every n from 1 to 32 (every group size G = 4, 8, 16, 32,
every shared-memory carve-up assign_smem_floats(n) and every bitonic padding size), on the tied, degenerate and extreme
cost families of test_lexifair_host.  For n <= 8 the oracle is brute force.  Above, lexifair_descent is the algorithm the
kernel mirrors, so every answer is also checked against an independent optimality certificate."""
import numpy as np
import pytest
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import maximum_bipartite_matching

from oracle.lexifair import lexifair_bruteforce_batched, lexifair_descent, rank_transform
from test_lexifair_host import cost_families

pytestmark = pytest.mark.gpu

THREADS = 128                                   # assign_kernel's CTA


@pytest.fixture(autouse=True)
def _mapping_independent(kernel_mapping):
    if kernel_mapping == "group":
        pytest.skip("the assignment entries do not depend on the kernel mapping: runs under 'auto' only")


def _group_size(n):
    return 4 if n <= 4 else 8 if n <= 8 else 16 if n <= 16 else 32


def _exact(costs):
    n = costs.shape[-1]
    return lexifair_bruteforce_batched(costs) if n <= 8 else np.stack([lexifair_descent(c) for c in costs])


def _certify(cost, pi):
    """pi is a permutation and the lexicographic-bottleneck optimum under the order (cost, i, j).  Walk pi from its largest
    key down: no perfect matching of the remaining rows / columns uses only keys below the current entry's, so every optimum
    of the remaining submatrix has that entry as its bottleneck and (keys being distinct) contains it; delete its row and
    column and go on."""
    n = cost.shape[0]
    assert sorted(pi.tolist()) == list(range(n)), pi
    key = rank_transform(cost)
    rows, cols = list(range(n)), list(range(n))
    for i in sorted(range(n), key=lambda r: -key[r, pi[r]]):
        k = key[i, pi[i]]
        sub = key[np.ix_(rows, cols)] < k
        if sub.any():
            m = maximum_bipartite_matching(csr_matrix(sub.astype(np.int8)), perm_type="column")
            assert (m >= 0).sum() < len(rows), (i, pi)
        rows.remove(i)
        cols.remove(int(pi[i]))


def _cdist(ap, gp):
    d = ap.astype(np.float64)[:, :, None, :] - gp.astype(np.float64)[:, None, :, :]
    return np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1])


def _check(got, costs, name):
    want = _exact(costs)
    bad = np.flatnonzero((got != want).any(1))
    assert bad.size == 0, (name, bad[:4], costs[bad[0]], got[bad[0]], want[bad[0]])
    if costs.shape[-1] > 8:
        for c, pi in zip(costs, got):
            _certify(c, pi)


@pytest.mark.parametrize("n", range(1, 33))
def test_every_n_matches_the_exact_oracle_on_every_family(n):
    import fair_marl_b200 as fm
    rng = np.random.default_rng(300 + n)
    num = 40 if n <= 8 else 5 if n <= 20 else 3
    fam, sigma = cost_families(rng, num, n)
    for name, costs in fam.items():
        got = fm.lexifair_batched(costs=costs)
        assert got.dtype == np.int32 and got.shape == (num, n)
        if name == "permutation":
            assert (got == sigma).all()
        _check(got, costs, name)
    ap = rng.uniform(-1, 1, (num, n, 2)).astype(np.float32)               # float32 positions -> float64 distances (cdist)
    gp = (0.8 * rng.uniform(-1, 1, (num, n, 2))).astype(np.float32)
    _check(fm.lexifair_batched(agent_pos=ap, goal_pos=gp), _cdist(ap, gp), "positions")


def _position_families(rng, num, n):
    fam = {}
    a = rng.uniform(-1, 1, (num, n, 2)).astype(np.float32)
    g = rng.uniform(-1, 1, (num, n, 2)).astype(np.float32)
    fam["coincident_agents"] = (np.broadcast_to(a[:, :1], a.shape).copy(), g)
    fam["coincident_goals"] = (a, np.broadcast_to(g[:, :1], g.shape).copy())
    on = rng.random((num, n)) < 0.6                                          # agents exactly on goals (distance 0)
    fam["agents_on_goals"] = (np.where(on[..., None], g[:, rng.permutation(n)], a), g)
    fam["grid_1_8"] = (rng.integers(-8, 9, (num, n, 2)).astype(np.float32) / 8,   # 3-4-5 triangles: exact distance ties
                       rng.integers(-8, 9, (num, n, 2)).astype(np.float32) / 8)
    return fam


@pytest.mark.parametrize("n", [2, 3, 4, 5, 7, 8, 9, 13, 16, 17, 24, 32])
def test_positions_with_exact_distance_ties(n):
    import fair_marl_b200 as fm
    rng = np.random.default_rng(400 + n)
    num = 60 if n <= 8 else 6
    for name, (ap, gp) in _position_families(rng, num, n).items():
        c = _cdist(ap, gp)
        assert any(np.unique(m).size < m.size for m in c), name
        _check(fm.lexifair_batched(agent_pos=ap, goal_pos=gp), c, name)


def test_grid_family_contains_3_4_5_ties():
    rng = np.random.default_rng(1)
    ap, gp = _position_families(rng, 200, 6)["grid_1_8"]
    c = _cdist(ap, gp)
    assert (c == 5 / 8).any() and ((c == 5 / 8) & (ap[:, :, None, 0] != gp[:, None, :, 0])
                                   & (ap[:, :, None, 1] != gp[:, None, :, 1])).any()


@pytest.mark.parametrize("n", [1, 3, 4, 5, 8, 9, 13, 16, 17, 29, 32])
def test_same_problem_in_every_slot_of_every_warp(n):
    """One tie-heavy problem copied into every group slot of a warp (EPW = 32 / G problems per warp) and every warp of the
    CTA, with a batch that ends in a partly filled warp: every copy gets the oracle's answer."""
    import fair_marl_b200 as fm
    G = _group_size(n)
    per_cta = (32 // G) * (THREADS // 32)
    num = 3 * per_cta + (32 // G) + 1 if G < 32 else 3 * per_cta + 1
    assert num % per_cta != 0
    rng = np.random.default_rng(500 + n)
    fam, _ = cost_families(rng, 1, n)
    for name in ("ties01", "ties012", "identical_rows", "last_ulp", "continuous"):
        one = fam[name]
        got = fm.lexifair_batched(costs=np.broadcast_to(one, (num, n, n)).copy())
        want = _exact(one)[0]
        assert (got == want).all(), (name, np.flatnonzero((got != want).any(1))[:8])


@pytest.mark.parametrize("n", [3, 5])
def test_large_batch_equals_each_problem_alone(n):
    """2^17 + 5 tie-heavy problems in one call: every answer equals brute force, and a sample solved one at a time gives the
    same bytes."""
    import torch
    import fair_marl_b200 as fm
    rng = np.random.default_rng(600 + n)
    num = (1 << 17) + 5
    costs = rng.integers(0, 3, (num, n, n)).astype(np.float64)
    costs[::3] = rng.random((len(costs[::3]), n, n))
    c = torch.as_tensor(costs, device="cuda")
    full = fm.lexifair_batched(costs=c)
    assert full.is_cuda and full.dtype == torch.int32
    assert (full.cpu().numpy() == lexifair_bruteforce_batched(costs)).all()
    for k in [0, 1, 7, 8, 31, 32, 127, 128, 4097, num - 2, num - 1] + rng.integers(0, num, 24).tolist():
        assert torch.equal(fm.lexifair_batched(costs=c[k:k + 1])[0], full[k]), k


def test_zero_problems_is_a_no_op():
    import torch
    import fair_marl_b200 as fm
    from fair_marl_b200 import _lib
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.fm_assign_costs(0, None, 0, 5, None, stream), "fm_assign_costs")
    _lib.check(lib.fm_assign_positions(0, None, None, 0, 5, None, stream), "fm_assign_positions")
    torch.cuda.synchronize()
    assert fm.lexifair_batched(costs=np.zeros((0, 5, 5))).shape == (0, 5)
    z = np.zeros((0, 4, 2), np.float32)
    assert fm.lexifair_batched(agent_pos=z, goal_pos=z).shape == (0, 4)
    with pytest.raises(fm._lib.FairMarlError):                       # a null pointer with work to do is still refused
        _lib.check(lib.fm_assign_costs(0, None, 1, 5, None, stream), "fm_assign_costs")


@pytest.mark.parametrize("n", [3, 7, 12, 32])
def test_non_finite_problem_gets_minus_one_rows_and_neighbours_are_unaffected(n):
    import fair_marl_b200 as fm
    rng = np.random.default_rng(700 + n)
    num = 70
    c = rng.integers(0, 3, (num, n, n)).astype(np.float64)
    clean = fm.lexifair_batched(costs=c)
    bad = {5: np.nan, 6: np.inf, 7: -np.inf, 40: np.nan, num - 1: np.inf}
    c2 = c.copy()
    for k, v in bad.items():
        c2[k, rng.integers(0, n), rng.integers(0, n)] = v
    c2[40, n - 1, 0] = np.inf
    got = fm.lexifair_batched(costs=c2)
    for k in range(num):
        if k in bad:
            assert (got[k] == -1).all(), k
        else:
            assert (got[k] == clean[k]).all(), k
    ap = rng.uniform(-1, 1, (6, n, 2)).astype(np.float32)
    gp = rng.uniform(-1, 1, (6, n, 2)).astype(np.float32)
    clean = fm.lexifair_batched(agent_pos=ap, goal_pos=gp)
    ap[1, n - 1, 0] = np.nan                                         # dist64 alone would turn a NaN coordinate into a distance of 0
    gp[2, 0, 1] = np.inf
    ap[4, 0, 1] = -np.inf
    got = fm.lexifair_batched(agent_pos=ap, goal_pos=gp)
    assert (got[[1, 2, 4]] == -1).all()
    assert (got[[0, 3, 5]] == clean[[0, 3, 5]]).all()


def test_solve_fair_assignment_raises_on_non_finite_costs_and_keeps_the_reference_instance():
    import fair_marl_b200 as fm
    goals = np.array([[0., -0.5], [0.45, -0.5], [0.9, -0.5]])
    agents = np.array([[-0.9, -0.9], [-0.9, 0.], [-0.9, 0.9]])
    d = np.sqrt(((agents[:, None, :] - goals[None, :, :]) ** 2).sum(-1))
    x, _ = fm.solve_fair_assignment(d)                                # marl_fair_assign.py:63-70
    assert (np.where(x == 1)[1] == [2, 1, 0]).all()
    for v in (np.nan, np.inf, -np.inf):
        e = d.copy()
        e[1, 2] = v
        with pytest.raises(ValueError):
            fm.solve_fair_assignment(e)
