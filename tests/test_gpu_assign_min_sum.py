"""Batched min-sum assignment on the GPU (fm_assign_min_sum_costs / fm_assign_min_sum_positions, csrc/fm_lsap.cu) against
scipy.optimize.linear_sum_assignment: col_ind bit for bit on every problem, tied optima included."""
import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

pytestmark = pytest.mark.gpu


def _scipy(costs):
    return np.stack([linear_sum_assignment(c)[1] for c in costs]).astype(np.int32)


def _costs(kind, rng, num, n):
    if kind == "random":
        return rng.random((num, n, n))
    if kind == "ties012":
        return rng.integers(0, 3, (num, n, n)).astype(np.float64)
    if kind == "wide_range":                                   # 1e-12 .. 1e12, log-uniform
        return 10.0 ** rng.uniform(-12, 12, (num, n, n))
    raise ValueError(kind)


@pytest.mark.parametrize("n", range(1, 33))
def test_min_sum_equals_scipy_for_every_n(n):
    import fair_marl_b200 as fm
    rng = np.random.default_rng(n)
    num = 96 if n <= 16 else 40
    for kind in ("random", "ties012", "wide_range"):
        c = _costs(kind, rng, num, n)
        got = fm.min_sum_batched(costs=c)
        assert got.dtype == np.int32 and got.shape == (num, n)
        ref = _scipy(c)
        bad = np.flatnonzero((got != ref).any(1))
        assert bad.size == 0, (kind, bad[:4], got[bad[:1]], ref[bad[:1]])
    a = rng.uniform(-1, 1, (num, n, 2)).astype(np.float32)        # float32 positions -> float64 distances (cdist)
    g = rng.uniform(-1, 1, (num, n, 2)).astype(np.float32)
    got = fm.min_sum_batched(agent_pos=a, goal_pos=g)
    d = np.sqrt(((a.astype(np.float64)[:, :, None] - g.astype(np.float64)[:, None]) ** 2).sum(-1))
    assert (got == _scipy(d)).all()


def test_problem_alone_equals_problem_inside_a_large_batch():
    import torch
    import fair_marl_b200 as fm
    rng = np.random.default_rng(3)
    n, num = 11, 50_000
    c = torch.as_tensor(rng.integers(0, 3, (num, n, n)).astype(np.float64), device="cuda")
    full = fm.min_sum_batched(costs=c)
    assert full.is_cuda and full.dtype == torch.int32
    for k in (0, 1, 4, 31_337, num - 1):
        alone = fm.min_sum_batched(costs=c[k:k + 1])
        assert torch.equal(alone[0], full[k]), k
        assert (full[k].cpu().numpy() == linear_sum_assignment(c[k].cpu().numpy())[1]).all(), k


def test_zero_problems_is_a_no_op():
    import torch
    import fair_marl_b200 as fm
    from fair_marl_b200 import _lib
    lib = _lib.load()
    out = torch.full((4,), 7, dtype=torch.int32, device="cuda")
    c = torch.zeros((1, 2, 2), dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.fm_assign_min_sum_costs(0, c.data_ptr(), 0, 2, out.data_ptr(), stream))
    p = torch.zeros((1, 2, 2), dtype=torch.float32, device="cuda")
    _lib.check(lib.fm_assign_min_sum_positions(0, p.data_ptr(), p.data_ptr(), 0, 2, out.data_ptr(), stream))
    torch.cuda.synchronize()
    assert (out == 7).all()
    assert fm.min_sum_batched(costs=np.zeros((0, 5, 5))).shape == (0, 5)


def test_non_finite_problem_gets_minus_one_rows_and_neighbours_are_unaffected():
    import fair_marl_b200 as fm
    rng = np.random.default_rng(9)
    n, num = 7, 64
    c = rng.random((num, n, n))
    c[5, 2, 3] = np.nan
    c[6, 0, 0] = np.inf
    c[7, 6, 1] = -np.inf
    c[40, 3, 3] = np.nan
    c[40, 1, 2] = np.inf
    got = fm.min_sum_batched(costs=c)
    bad = {5, 6, 7, 40}
    for k in range(num):
        if k in bad:
            assert (got[k] == -1).all(), k
        else:
            assert (got[k] == linear_sum_assignment(c[k])[1]).all(), k
    pos = rng.uniform(-1, 1, (3, n, 2)).astype(np.float32)
    goal = pos[:, ::-1].copy()
    pos[1, 4, 0] = np.nan                                  # dist64 alone would turn a NaN coordinate into a distance of 0
    goal[2, 0, 1] = np.inf
    got = fm.min_sum_batched(agent_pos=pos, goal_pos=goal)
    assert (got[1:] == -1).all() and (got[0] == np.arange(n)[::-1]).all()


def test_captured_in_a_cuda_graph():
    import torch
    from fair_marl_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(4)
    n, num = 20, 300
    c = torch.as_tensor(rng.random((num, n, n)), device="cuda")
    out = torch.empty((num, n), dtype=torch.int32, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            _lib.check(lib.fm_assign_min_sum_costs(0, c.data_ptr(), num, n, out.data_ptr(), s.cuda_stream))
    torch.cuda.synchronize()
    for rep in range(2):
        c.copy_(torch.as_tensor(rng.random((num, n, n)), device="cuda"))
        out.fill_(-7)
        graph.replay()
        torch.cuda.synchronize()
        assert (out.cpu().numpy() == _scipy(c.cpu().numpy())).all(), rep


def test_linear_sum_assignment_is_a_drop_in_for_scipy():
    import fair_marl_b200 as fm
    rng = np.random.default_rng(12)
    for n in (1, 2, 5, 7, 16, 32):
        for c in (rng.random((n, n)), rng.integers(0, 2, (n, n)), rng.integers(0, 3, (n, n)).tolist()):
            r, k = fm.linear_sum_assignment(c)
            rr, rk = linear_sum_assignment(np.asarray(c, dtype=np.float64))
            assert r.dtype == np.int64 and k.dtype == np.int64
            assert (r == rr).all() and (k == rk).all()
    with pytest.raises(ValueError):
        fm.linear_sum_assignment(rng.random((3, 4)))
    with pytest.raises(ValueError):
        fm.linear_sum_assignment(np.full((3, 3), np.nan))
