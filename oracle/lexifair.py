"""Exact CPU solvers for the "lexifair" goal assignment (TEST INFRASTRUCTURE ONLY).

Reference: ``marl_fair_assign.py:16-55`` (``solve_fair_assignment``), called
from ``multiagent/custom_scenarios/navigation_graph.py:555-561``.

The reference solves n rounds of a binary MILP with pyomo + ``gurobi_persistent``
(neither vendored in the original project nor installable here; requirements.txt:2
pins gurobipy==10.0.2, pyomo is unpinned).  Round k: minimise z subject to
``cost_helper[i,j] * x[i,j] <= z`` over perfect matchings x, with the rows fixed
in earlier rounds held; then the entry of ``costs`` closest to the optimum z is
located (``np.argmin(np.abs(costs - obj))``, :39), its ``cost_helper`` is zeroed
and its row is frozen to the current assignment (:42, :50-52).

Published algorithm restated: at the optimum of a min-max ("bottleneck")
matching problem with distinct costs, the entry attaining z* is contained in
EVERY optimal matching (otherwise a matching with a smaller maximum would
exist), so freezing its row is independent of which optimal x the solver
returned, and the n rounds produce the unique assignment whose descending-sorted
cost vector is lexicographically minimal: the lexicographic bottleneck
assignment.  ``lexifair_milp`` restates the MILP sequence literally on HiGHS
(``scipy.optimize.milp``); ``lexifair_bruteforce`` enumerates permutations;
``lexifair_descent`` is the threshold-descent algorithm the CUDA kernel mirrors.

Parity: unpinned against Gurobi itself (not available).  Pinned against the one
fixed instance the reference carries (marl_fair_assign.py:63-64 -> [2, 1, 0])
and cross-checked between the three solvers in tests/test_oracle_lexifair.py.

Tie-break (exact cost ties have probability ~0 for continuous random positions;
the reference's behaviour under ties is solver dependent): entries are totally
ordered by ``(cost, agent index i, goal index j)``; all solvers here, and the
CUDA kernel, work on that order.
"""
from __future__ import annotations

import itertools
from functools import lru_cache

import numpy as np

__all__ = [
    "rank_transform",
    "lexifair_bruteforce",
    "lexifair_bruteforce_batched",
    "lexifair_descent",
    "lexifair_milp",
    "lexifair",
    "solve_fair_assignment",
]


def rank_transform(costs: np.ndarray) -> np.ndarray:
    """Replace every cost by its rank in the total order (cost, i, j).

    costs: [..., n, n] float.  Returns int64 ranks in [0, n*n), all distinct per
    matrix.  A stable argsort of the row-major flattened matrix realises the
    (cost, i, j) order because the flat index is i*n + j.
    """
    c = np.asarray(costs)
    n = c.shape[-1]
    flat = c.reshape(c.shape[:-2] + (n * n,))
    order = np.argsort(flat, axis=-1, kind="stable")
    ranks = np.empty_like(order)
    np.put_along_axis(ranks, order, np.broadcast_to(np.arange(n * n), order.shape), axis=-1)
    return ranks.reshape(c.shape).astype(np.int64)


@lru_cache(maxsize=None)
def _perms(n: int) -> np.ndarray:
    return np.array(list(itertools.permutations(range(n))), dtype=np.int64)


def lexifair_bruteforce(costs: np.ndarray) -> np.ndarray:
    """Lexicographic-min of the descending-sorted cost vector over all n! permutations.

    costs [n, n] -> goal index per agent, int64 [n].  n <= 9.
    """
    return lexifair_bruteforce_batched(np.asarray(costs)[None])[0]


def lexifair_bruteforce_batched(costs: np.ndarray) -> np.ndarray:
    """Batched brute force.  costs [B, n, n] -> [B, n] int64.  Needs n*n <= 64, n <= 8.

    The descending-sorted rank vector (ranks < n*n <= 64, 6 bits each) is packed
    into one integer, most significant = largest rank, so lexicographic order of
    the vectors is numeric order of the packed keys.
    """
    c = np.asarray(costs)
    B, n, _ = c.shape
    assert n <= 8, "brute force packs ranks into 6-bit fields"
    ranks = rank_transform(c)                                  # [B, n, n]
    perms = _perms(n)                                          # [P, n]
    rows = np.arange(n)
    out = np.empty((B, n), dtype=np.int64)
    chunk = max(1, (1 << 22) // (perms.shape[0] * n))
    shifts = (6 * np.arange(n - 1, -1, -1)).astype(np.uint64)  # largest rank most significant
    for s in range(0, B, chunk):
        r = ranks[s:s + chunk][:, rows[None, :], perms]        # [b, P, n] rank of (i, perm[i])
        r = -np.sort(-r, axis=-1)                              # descending
        key = (r.astype(np.uint64) << shifts).sum(axis=-1, dtype=np.uint64)
        best = np.argmin(key, axis=-1)
        out[s:s + chunk] = perms[best]
    return out


def lexifair_descent(costs: np.ndarray) -> np.ndarray:
    """Threshold descent: any n.  costs [n, n] -> [n] int64.

    Visit entries from the largest key down.  Delete the entry; if the bipartite
    graph of the remaining entries (restricted to rows / columns not yet frozen)
    still has a perfect matching, the deletion stands.  Otherwise the entry is
    the bottleneck of every remaining solution: restore it, freeze its row and
    column (this is the reference's "fix row r", marl_fair_assign.py:50-52) and
    continue.  The CUDA kernel (fair-marl_b200/csrc) follows the same steps with
    bit-mask rows.
    """
    c = np.asarray(costs)
    n = c.shape[0]
    ranks = rank_transform(c)
    order = np.argsort(-ranks.reshape(-1), kind="stable")      # descending key
    present = np.ones((n, n), dtype=bool)
    row_match = np.arange(n)                                   # identity is a perfect matching
    col_match = np.arange(n)
    row_fixed = np.zeros(n, dtype=bool)
    col_fixed = np.zeros(n, dtype=bool)

    def try_row(i: int, seen: np.ndarray) -> bool:
        for cc in range(n):
            if not present[i, cc] or col_fixed[cc] or seen[cc]:
                continue
            seen[cc] = True
            if col_match[cc] < 0 or try_row(int(col_match[cc]), seen):
                col_match[cc] = i
                row_match[i] = cc
                return True
        return False

    for flat in order:
        i, j = divmod(int(flat), n)
        if row_fixed[i] or col_fixed[j]:
            continue
        present[i, j] = False
        if row_match[i] != j:
            continue
        col_match[j] = -1
        row_match[i] = -1
        if try_row(i, np.zeros(n, dtype=bool)):
            continue
        present[i, j] = True
        row_match[i] = j
        col_match[j] = i
        row_fixed[i] = True
        col_fixed[j] = True
    assert row_fixed.all()
    return row_match.astype(np.int64)


def lexifair_milp(costs: np.ndarray):
    """Literal HiGHS restatement of marl_fair_assign.py:16-55.  Returns (x, objs).

    Same variables (x binary n*nj, z free), same constraints (coverage :12,
    assignment :13, aux :25 rebuilt every round :44-49, assigned rows :50-52),
    same ``argmin |costs - obj|`` row selection (:39).
    """
    from scipy.optimize import Bounds, LinearConstraint, milp

    costs = np.asarray(costs, dtype=np.float64)
    n, nj = costs.shape
    nx = n * nj
    cost_helper = costs.copy()
    obj = np.zeros(nx + 1)
    obj[-1] = 1.0
    integrality = np.concatenate([np.ones(nx), [0.0]])
    lb = np.concatenate([np.zeros(nx), [-np.inf]])
    ub = np.concatenate([np.ones(nx), [np.inf]])
    a_cov = np.zeros((nj, nx + 1))
    for j in range(nj):
        a_cov[j, [i * nj + j for i in range(n)]] = 1.0
    a_asg = np.zeros((n, nx + 1))
    for i in range(n):
        a_asg[i, i * nj:(i + 1) * nj] = 1.0
    fixed = []                                     # (variable index, value)
    x = None
    for _ in range(n):
        a_aux = np.zeros((nx, nx + 1))
        a_aux[np.arange(nx), np.arange(nx)] = cost_helper.reshape(-1)
        a_aux[:, -1] = -1.0
        cons = [LinearConstraint(a_cov, 1.0, 1.0), LinearConstraint(a_asg, 1.0, 1.0),
                LinearConstraint(a_aux, -np.inf, 0.0)]
        lo, hi = lb.copy(), ub.copy()
        for k, v in fixed:
            lo[k] = hi[k] = v
        res = milp(obj, constraints=cons, integrality=integrality, bounds=Bounds(lo, hi))
        assert res.status == 0, res.message
        x = np.rint(res.x[:nx]).reshape(n, nj).astype(int)
        z = res.x[-1]
        r, c = np.unravel_index(np.argmin(np.abs(costs - z)), (n, nj))
        cost_helper[r, c] = 0.0
        for j in range(nj):
            fixed.append((r * nj + j, float(x[r, j])))
    objs = np.sort(np.sum(costs * x, axis=1))[::-1]
    return x, objs


def lexifair(costs: np.ndarray) -> np.ndarray:
    """costs [B, n, n] or [n, n] -> goal index per agent."""
    c = np.asarray(costs)
    if c.ndim == 2:
        return lexifair(c[None])[0]
    n = c.shape[-1]
    if n <= 7:
        return lexifair_bruteforce_batched(c)
    return np.stack([lexifair_descent(m) for m in c])


def solve_fair_assignment(costs: np.ndarray):
    """Drop-in for ``marl_fair_assign.solve_fair_assignment`` (same return convention:
    ``x`` 0/1 int matrix and descending per-agent costs, marl_fair_assign.py:54-55).
    Registered as the ``marl_fair_assign`` module stub by ``reference_shim``.
    """
    costs = np.asarray(costs, dtype=np.float64)
    n = costs.shape[0]
    match = lexifair(costs)
    x = np.zeros((n, n), dtype=int)
    x[np.arange(n), match] = 1
    objs = np.sort(np.sum(costs * x, axis=1))[::-1]
    return x, objs
