"""The per-thread min-sum solver of csrc/fm_form.cuh (f_min_sum_sap, formation OA at N >= 6) compiled for the host (g++,
ASan + UBSan, -ffp-contract=off) and checked against scipy.optimize.linear_sum_assignment on tie-heavy matrices, then
the whole OA reset + rollout at N = 6 and 7 against the oracle through the host build of test_kernel_source_host.  Test
infrastructure: not a CPU path of the product."""
import os
import subprocess

import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

from oracle.formation import FormationConfig, FormationOracle
from test_kernel_source_host import CSRC, EMUL, ROOT, _compare, _run, host_exe  # noqa: F401  (host_exe: a fixture)

_MAIN = r"""
template <int N>
static void solve(FILE* f, FILE* g, int num) {
  std::vector<double> c(N * N);
  for (int p = 0; p < num; ++p) {
    if (fread(c.data(), 8, N * N, f) != (size_t)(N * N)) exit(5);
    int m[N]; double d[N];
    fm::f_min_sum_sap<N>(c.data(), m, d);
    fwrite(m, 4, N, g); fwrite(d, 8, N, g);
  }
}
int main(int argc, char** argv) {
  if (argc != 3) return 2;
  FILE* f = fopen(argv[1], "rb"); FILE* g = fopen(argv[2], "wb");
  if (!f || !g) return 3;
  int32_t h[2];
  if (fread(h, 4, 2, f) != 2) return 4;
  switch (h[1]) {
    case 1: solve<1>(f, g, h[0]); break; case 2: solve<2>(f, g, h[0]); break; case 3: solve<3>(f, g, h[0]); break;
    case 4: solve<4>(f, g, h[0]); break; case 5: solve<5>(f, g, h[0]); break; case 6: solve<6>(f, g, h[0]); break;
    case 7: solve<7>(f, g, h[0]); break; case 8: solve<8>(f, g, h[0]); break;
    default: return 6;
  }
  fclose(f); fclose(g);
  return 0;
}
"""


@pytest.fixture(scope="module")
def solver_exe(tmp_path_factory):
    form = open(os.path.join(CSRC, "fm_form.cuh")).read()
    a = form.index("template <int N>\n__device__ __noinline__ void f_min_sum_sap(")
    body = form[a:form.index("template <int N>\n__device__ __forceinline__ void f_min_sum(", a)]
    src = "\n".join(['#include "prelude.h"', "namespace fm {", body, "}  // namespace fm", _MAIN])
    d = tmp_path_factory.mktemp("min_sum_host")
    cpp, exe = d / "min_sum_host.cpp", d / "min_sum_host"
    cpp.write_text(src)
    cmd = ["g++", "-std=c++17", "-O1", "-g", "-ffp-contract=off", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
           "-ftrivial-auto-var-init=pattern", "-I", EMUL, "-I", os.path.join(ROOT, "include"), str(cpp), "-o", str(exe)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]
    return str(exe)


def _solve(exe, tmp, costs):
    num, n = costs.shape[0], costs.shape[1]
    fin, fout = os.path.join(tmp, "in.bin"), os.path.join(tmp, "out.bin")
    with open(fin, "wb") as f:
        np.array([num, n], np.int32).tofile(f)
        np.ascontiguousarray(costs, dtype=np.float64).tofile(f)
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0", UBSAN_OPTIONS="print_stacktrace=1")
    res = subprocess.run([exe, fin, fout], capture_output=True, text=True, env=env)
    assert res.returncode == 0, res.stderr[-4000:]
    raw = np.fromfile(fout, np.uint8).reshape(num, n * 12)
    return raw[:, :4 * n].copy().view(np.int32), raw[:, 4 * n:].copy().view(np.float64)


def _tie_heavy(rng, num, n):
    """Four kinds of cost: integer ties in {0, 1} and {0, 1, 2}, random float64, float64 distances of float32 points."""
    c = np.empty((num, n, n))
    k = num // 4
    c[:k] = rng.integers(0, 2, (k, n, n))
    c[k:2 * k] = rng.integers(0, 3, (k, n, n))
    c[2 * k:3 * k] = rng.random((k, n, n))
    a = rng.uniform(-1, 1, (num - 3 * k, n, 2)).astype(np.float32).astype(np.float64)
    g = rng.uniform(-1, 1, (num - 3 * k, n, 2)).astype(np.float32).astype(np.float64)
    c[3 * k:] = np.sqrt(((a[:, :, None] - g[:, None]) ** 2).sum(-1))
    return c


@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7])
def test_per_thread_solver_equals_scipy(solver_exe, tmp_path, n):
    rng = np.random.default_rng(40 + n)
    costs = _tie_heavy(rng, 800, n)
    match, delta = _solve(solver_exe, str(tmp_path), costs)
    for p in range(costs.shape[0]):
        ref = linear_sum_assignment(costs[p])[1]
        assert (match[p] == ref).all(), (p, costs[p], match[p], ref)
        assert (delta[p] == costs[p][np.arange(n), ref]).all(), p


@pytest.mark.parametrize("N,O", [(6, 0), (6, 2), (7, 1), (7, 3)])
def test_oa_reset_and_rollout_source_matches_oracle(host_exe, tmp_path, N, O):  # noqa: F811
    """OA at N = 6 and 7 (f_min_sum_sap in the reset and in agent 0's reward call): reset bit for bit, then 12 goal-seeking
    steps with auto-resets, every output and the state against the oracle (which calls scipy)."""
    B = 24
    cfg = FormationConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=8,
                          fairness_reward=False, assignment="optimal")
    orc = FormationOracle(cfg, B, seed=7, env_offset=3)
    ref = orc.reset()
    zero = FormationOracle(cfg, B).get_state()
    for name in ("dists_to_goal", "times_required", "dist_left_to_goal", "goal_reached", "goal_history"):
        getattr(zero, name)[:] = 0.0
    zero.min_time[:] = 0.0
    out, st = _run(host_exe, str(tmp_path), cfg, zero, is_reset=True, seed=7, env_offset=3)
    rs = orc.get_state()
    for f in ("pos", "landmark_pos", "obstacle_pos", "goal_match", "episode"):
        assert (getattr(st, f) == getattr(rs, f)).all(), f
    rng = np.random.default_rng(5)
    resets = 0
    for t in range(12):
        orc.set_state(st)
        d = np.take_along_axis(st.landmark_pos, st.goal_match[..., None], axis=1) - st.pos
        seek = np.where(np.abs(d[..., 0]) > np.abs(d[..., 1]), np.where(d[..., 0] > 0, 1, 2), np.where(d[..., 1] > 0, 3, 4))
        a = np.where(rng.random((B, N)) < 0.25, rng.integers(0, 5, (B, N)), seek)
        out, st = _run(host_exe, str(tmp_path), cfg, st, actions=a, seed=7, env_offset=3, auto_reset=True)
        ref = orc.step(a, autoreset=True)
        _compare(out, ref, st, orc.get_state())
        resets += int(ref["reset"].sum())
    assert resets >= B
