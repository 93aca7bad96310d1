"""Batched goal assignment on the GPU: lexifair, drop-in for ``marl_fair_assign.solve_fair_assignment``
(marl_fair_assign.py:16-55; call site navigation_graph.py:555-561), and min-sum, drop-in for
``scipy.optimize.linear_sum_assignment`` on square matrices (nav_base_formation_graph_mask.py:255-260)."""
from __future__ import annotations

import numpy as np

from fair_marl_b200 import _lib


def _batched(entry_costs: str, entry_positions: str, costs, agent_pos, goal_pos, device: int):
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = torch.device("cuda", device)
    stream = torch.cuda.current_stream(dev).cuda_stream
    as_numpy = isinstance(costs if costs is not None else agent_pos, np.ndarray)
    with torch.cuda.device(dev):
        if costs is not None:
            c = torch.as_tensor(costs, dtype=torch.float64, device=dev).contiguous()
            if c.dim() != 3 or c.shape[1] != c.shape[2]:
                raise ValueError(f"costs must be [num, n, n], got {tuple(c.shape)}")
            num, n = int(c.shape[0]), int(c.shape[1])
            out = torch.empty((num, n), dtype=torch.int32, device=dev)
            _lib.check(getattr(lib, entry_costs)(device, c.data_ptr(), num, n, out.data_ptr(), stream), entry_costs)
        else:
            a = torch.as_tensor(agent_pos, dtype=torch.float32, device=dev).contiguous()
            g = torch.as_tensor(goal_pos, dtype=torch.float32, device=dev).contiguous()
            if a.shape != g.shape or a.dim() != 3 or a.shape[2] != 2:
                raise ValueError("agent_pos / goal_pos must both be [num, n, 2]")
            num, n = int(a.shape[0]), int(a.shape[1])
            out = torch.empty((num, n), dtype=torch.int32, device=dev)
            _lib.check(getattr(lib, entry_positions)(device, a.data_ptr(), g.data_ptr(), num, n, out.data_ptr(), stream),
                       entry_positions)
    return out.cpu().numpy() if as_numpy else out


def lexifair_batched(costs=None, agent_pos=None, goal_pos=None, device: int = 0):
    """Goal index per agent for a batch of problems, computed on the GPU.

    Either ``costs`` [num, n, n] (float64; torch CUDA tensor or numpy) or ``agent_pos`` / ``goal_pos``
    [num, n, 2] float32 (costs = float64 Euclidean distances, ``cdist``).  Returns an int32 torch CUDA
    tensor [num, n] when given tensors, a numpy array when given numpy.  Entries are ordered by
    (cost, agent, goal), so tied costs have one answer, the oracle's.  A problem with any NaN or +-inf
    cost (or coordinate) gets -1 in every entry of its row; ``num == 0`` is allowed.
    """
    return _batched("fm_assign_costs", "fm_assign_positions", costs, agent_pos, goal_pos, device)


def min_sum_batched(costs=None, agent_pos=None, goal_pos=None, device: int = 0):
    """Min-sum matching per problem for a batch, computed on the GPU: ``out[p]`` equals
    ``scipy.optimize.linear_sum_assignment(costs[p])[1]`` bit for bit, ties included.

    Inputs and return type as ``lexifair_batched``; n <= 32.  A problem with any NaN or +-inf cost gets -1 in
    every entry of its row.
    """
    return _batched("fm_assign_min_sum_costs", "fm_assign_min_sum_positions", costs, agent_pos, goal_pos, device)


def linear_sum_assignment(cost_matrix):
    """Drop-in for ``scipy.optimize.linear_sum_assignment(cost_matrix)`` on a square matrix (minimise), solved on the
    GPU: ``(row_ind, col_ind)`` as numpy int64, equal to scipy's.  A non-square matrix raises ``ValueError``; so does
    a matrix with NaN or +-inf entries."""
    c = np.asarray(cost_matrix, dtype=np.float64)
    if c.ndim != 2 or c.shape[0] != c.shape[1]:
        raise ValueError(f"square cost matrix expected, got shape {c.shape}")
    n = c.shape[0]
    if n == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    col = min_sum_batched(costs=c[None])[0]
    if (col < 0).any():
        raise ValueError("cost matrix contains NaN or infinite entries")
    return np.arange(n, dtype=np.int64), col.astype(np.int64)


def solve_fair_assignment(costs):
    """Same signature and return convention as the reference function: ``(x, objs)`` with ``x`` the
    0/1 int assignment matrix and ``objs`` the per-agent costs sorted descending
    (marl_fair_assign.py:54-55).  A matrix with NaN or +-inf entries raises ``ValueError``."""
    costs = np.asarray(costs, dtype=np.float64)
    assert np.ndim(costs) == 2                      # marl_fair_assign.py:6
    n, nj = costs.shape
    if n != nj:
        raise ValueError("square cost matrix expected (num_agents == num_landmarks)")
    match = lexifair_batched(costs=costs[None])[0]
    if (match < 0).any():
        raise ValueError("cost matrix contains NaN or infinite entries")
    x = np.zeros((n, nj), dtype=int)
    x[np.arange(n), match] = 1
    objs = np.sort(np.sum(costs * x, axis=1))[::-1]
    return x, objs


def pair_dist(a, b, device: int = 0):
    """float64 ``||a[k] - b[k]||`` for float32 points ``a``, ``b`` [num, 2] with the kernels' distance
    primitive (``fm_pair_dist``): bit-identical to ``np.linalg.norm(a64 - b64, axis=1)`` evaluated as
    sqrt(dx*dx + dy*dy) in float64 (core.py:204-228, navigation_graph.py:555)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = torch.device("cuda", device)
    as_numpy = isinstance(a, np.ndarray)
    with torch.cuda.device(dev):
        ta = torch.as_tensor(a, dtype=torch.float32, device=dev).contiguous()
        tb = torch.as_tensor(b, dtype=torch.float32, device=dev).contiguous()
        if ta.shape != tb.shape or ta.dim() != 2 or ta.shape[1] != 2:
            raise ValueError("a / b must both be [num, 2]")
        out = torch.empty(ta.shape[0], dtype=torch.float64, device=dev)
        _lib.check(lib.fm_pair_dist(device, ta.data_ptr(), tb.data_ptr(), int(ta.shape[0]), out.data_ptr(),
                                    torch.cuda.current_stream(dev).cuda_stream), "fm_pair_dist")
    return out.cpu().numpy() if as_numpy else out
