"""The min-sum assignment without a GPU: the readable statement of the solver's contract (oracle/lsap.py) against scipy,
and the new entry points' argument checks, which come before any device call."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

from oracle.lsap import lsap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tie_heavy(rng, n, k):
    kind = k % 4
    if kind == 0:
        return rng.integers(0, 2, (n, n)).astype(np.float64)
    if kind == 1:
        return rng.integers(0, 3, (n, n)).astype(np.float64)
    if kind == 2:
        return rng.random((n, n))
    a = rng.uniform(-1, 1, (n, 2)).astype(np.float32).astype(np.float64)
    g = rng.uniform(-1, 1, (n, 2)).astype(np.float32).astype(np.float64)
    return np.sqrt(((a[:, None] - g[None]) ** 2).sum(-1))


@pytest.mark.parametrize("n", range(1, 33))
def test_oracle_lsap_equals_scipy_on_tie_heavy_matrices(n):
    """Both forms of the column choice (scipy's sequential scan, and the one-reduction key a warp computes) give scipy's
    col_ind on every matrix, the many tied optima of the {0, 1} and {0, 1, 2} matrices included."""
    rng = np.random.default_rng(1000 + n)
    for k in range(24 if n <= 16 else 8):
        c = _tie_heavy(rng, n, k)
        ref = linear_sum_assignment(c)[1]
        assert (lsap(c) == ref).all(), (k, c)
        assert (lsap(c, reduction=True) == ref).all(), (k, c)


def test_oracle_lsap_rejects_non_square():
    with pytest.raises(ValueError):
        lsap(np.zeros((2, 3)))


@pytest.fixture(scope="module")
def lib():
    import fair_marl_b200
    fair_marl_b200.build_library()
    from fair_marl_b200 import _lib
    return _lib.load()


@pytest.mark.parametrize("entry", ["fm_assign_min_sum_costs", "fm_assign_min_sum_positions"])
def test_min_sum_entries_reject_bad_arguments_before_the_device(lib, entry):
    """n = 0, n = 33, a null pointer and num < 0 are argument errors (-1) whether or not a device is present."""
    buf = (ctypes.c_double * 64)()
    out = (ctypes.c_int32 * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    o = ctypes.cast(out, ctypes.c_void_p)
    fn = getattr(lib, entry)

    def call(num, n, inp=p, dst=o):
        if entry.endswith("costs"):
            return fn(0, inp, num, n, dst, None)
        return fn(0, inp, inp, num, n, dst, None)

    assert call(1, 0) == -1 and b"n must be in 1..32" in lib.fm_last_error()
    assert call(1, 33) == -1 and b"(got 33)" in lib.fm_last_error()
    assert call(1, 3, inp=None) == -1 and b"null" in lib.fm_last_error()
    assert call(1, 3, dst=None) == -1 and b"null" in lib.fm_last_error()
    assert call(-1, 3) == -1 and b"num < 0" in lib.fm_last_error()


_NO_DEVICE = """
import numpy as np
import fair_marl_b200 as fm
from fair_marl_b200 import _lib
for call in (lambda: fm.min_sum_batched(costs=np.zeros((2, 3, 3))),
             lambda: fm.min_sum_batched(agent_pos=np.zeros((2, 3, 2), np.float32), goal_pos=np.zeros((2, 3, 2), np.float32)),
             lambda: fm.linear_sum_assignment(np.eye(3))):
    try:
        call()
        raise SystemExit("min-sum assignment computed without a CUDA device")
    except _lib.FairMarlError:
        pass
"""


def test_min_sum_batched_raises_without_a_device(lib):
    """In a child process that sees no CUDA device, so the check holds on GPU machines too."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", _NO_DEVICE], cwd=ROOT, env=env, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr


def test_linear_sum_assignment_rejects_non_square():
    import fair_marl_b200 as fm
    with pytest.raises(ValueError):
        fm.linear_sum_assignment(np.zeros((2, 3)))
