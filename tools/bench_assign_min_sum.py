#!/usr/bin/env python
"""Batched min-sum assignment alone (fm_assign_min_sum_positions, csrc/fm_lsap.cu: one warp per problem), against
scipy.optimize.linear_sum_assignment on one CPU core.
usage: python tools/bench_assign_min_sum.py   (on the GPU box) -> one JSON line per n"""
import json, os, sys, time
import numpy as np, torch
from scipy.optimize import linear_sum_assignment
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import fair_marl_b200 as fm  # noqa: E402,F401
from fair_marl_b200 import _lib  # noqa: E402

lib = _lib.load()
dev = torch.device("cuda", 0)
props = torch.cuda.get_device_properties(dev)
for n, num in ((3, 65536), (7, 262144), (16, 131072), (32, 32768)):
    g = torch.Generator(device=dev).manual_seed(n)
    a = (torch.rand((num, n, 2), generator=g, device=dev) * 2 - 1).float()
    l = ((torch.rand((num, n, 2), generator=g, device=dev) * 2 - 1) * 0.8).float()
    out = torch.empty((num, n), dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    for _ in range(3):
        _lib.check(lib.fm_assign_min_sum_positions(0, a.data_ptr(), l.data_ptr(), num, n, out.data_ptr(), st))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    e0.record()
    for _ in range(reps):
        _lib.check(lib.fm_assign_min_sum_positions(0, a.data_ptr(), l.data_ptr(), num, n, out.data_ptr(), st))
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    # scipy on a sample of the same problems, one core
    k = 4000 if n <= 7 else 1000
    aa, ll = a[:k].cpu().numpy().astype(np.float64), l[:k].cpu().numpy().astype(np.float64)
    d = aa[:, :, None, :] - ll[:, None, :, :]
    costs = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1])
    t0 = time.perf_counter(); ref = np.stack([linear_sum_assignment(c)[1] for c in costs]); t1 = time.perf_counter()
    ok = bool((out[:k].cpu().numpy() == ref).all())
    print(json.dumps({"kernel": "lsap_kernel (fm_assign_min_sum_positions)", "gpu": props.name, "n": n, "problems": num,
                      "ms_per_call": ms, "solves_per_s": num / (ms * 1e-3), "bit_exact_vs_scipy_sample": ok,
                      "scipy_solves_per_s_1core": k / (t1 - t0)}), flush=True)
