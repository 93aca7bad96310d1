"""Min-sum assignment by shortest augmenting paths, as scipy computes it (TEST INFRASTRUCTURE ONLY).

Reference: ``scipy.optimize.linear_sum_assignment`` (``scipy/optimize/rectangular_lsap/rectangular_lsap.cpp``, after
D. F. Crouse, "On implementing 2D rectangular assignment algorithms", IEEE TAES 52(4), 2016), square case, minimise.
The original project calls it in the optimal-assignment formation scenario (nav_base_formation_graph_mask.py:255-260,
:686-689).

This is the readable statement of the contract the CUDA solvers follow (``f_min_sum_sap`` in csrc/fm_form.cuh,
``lsap_kernel`` in csrc/fm_lsap.cu): scipy's operation order and its tie rule, so that the matching equals scipy's
``col_ind`` bit for bit, also when several matchings tie for the optimum.  The reduced cost of a column is
``minVal + cost[i][j] - u[i] - v[j]`` in float64, left to right.  Among the remaining columns the one of smallest
``spc`` is taken; among equal values a later column in ``remaining`` replaces an earlier one only if it is unassigned.

``argmin_key`` is the same choice as one reduction, which is what a warp computes: the smallest ``spc``; among columns
at that value the unassigned one of LARGEST position in ``remaining`` if there is one, else the assigned one of
SMALLEST position.
"""
from __future__ import annotations

import numpy as np

__all__ = ["lsap", "argmin_key"]


def argmin_key(spc, remaining, nrem, row4col) -> int:
    """Position in ``remaining`` of the column scipy's scan picks, computed as a reduction."""
    best, best_key = -1, None
    for it in range(nrem):
        j = remaining[it]
        tie = (nrem - it) if row4col[j] == -1 else (32 + 1 + it)     # smaller is better
        key = (spc[j], tie)
        if best_key is None or key < best_key:
            best, best_key = it, key
    return best


def lsap(cost, reduction: bool = False) -> np.ndarray:
    """col4row of the square float64 matrix ``cost``: agent i -> goal ``col4row[i]`` (scipy's ``col_ind``).

    ``reduction=True`` picks the column with ``argmin_key`` instead of the sequential scan (same result)."""
    cost = np.asarray(cost, dtype=np.float64)
    n = cost.shape[0]
    if cost.ndim != 2 or cost.shape[1] != n:
        raise ValueError(f"square cost matrix expected, got {cost.shape}")
    u, v = np.zeros(n), np.zeros(n)
    col4row, row4col, path = [-1] * n, [-1] * n, [-1] * n
    for cur in range(n):
        min_val = 0.0
        remaining = [n - 1 - it for it in range(n)]
        nrem = n
        sr, sc = [False] * n, [False] * n
        spc = [np.inf] * n
        i, sink = cur, -1
        while sink == -1:
            sr[i] = True
            if reduction:
                for it in range(nrem):
                    j = remaining[it]
                    r = min_val + cost[i, j] - u[i] - v[j]
                    if r < spc[j]:
                        path[j], spc[j] = i, r
                index = argmin_key(spc, remaining, nrem, row4col)
                lowest = spc[remaining[index]]
            else:
                index, lowest = -1, np.inf
                for it in range(nrem):
                    j = remaining[it]
                    r = min_val + cost[i, j] - u[i] - v[j]
                    if r < spc[j]:
                        path[j], spc[j] = i, r
                    if spc[j] < lowest or (spc[j] == lowest and row4col[j] == -1):
                        lowest, index = spc[j], it
            min_val = lowest
            j = remaining[index]
            if row4col[j] == -1:
                sink = j
            else:
                i = row4col[j]
            sc[j] = True
            nrem -= 1
            remaining[index] = remaining[nrem]
        u[cur] += min_val
        for i in range(n):
            if sr[i] and i != cur:
                u[i] += min_val - spc[col4row[i]]
        for j in range(n):
            if sc[j]:
                v[j] -= min_val - spc[j]
        j = sink
        while True:
            i = path[j]
            row4col[j] = i
            col4row[i], j = j, col4row[i]
            if i == cur:
                break
    return np.asarray(col4row, dtype=np.int64)
