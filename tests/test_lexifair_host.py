"""The two per-thread lexifair solvers compiled for the host (g++, ASan + UBSan, -ffp-contract=off) and checked bit for bit
against the brute-force oracle on tied, degenerate and extreme costs:
  * lexifair_small<N> (csrc/fm_small.cuh, N <= 4, enumeration on rank keys): agent-warp resets, the formation logic and
    fused kernels at N <= 4;
  * lexifair_serial<N> (csrc/fm_form.cuh, N <= 8, sorted descent with a depth-first search): the formation fused kernel at
    N = 5 ... 7, every step.
Both must follow the total order (cost, i, j) of oracle/lexifair.py, ties included.  Continuous positions almost never tie,
so the rollout tests cannot tell a wrong tie rule from the right one; these families can.  FM_HOST_EMUL_CSRC points the
build at another source tree (as for test_kernel_source_host).  Test infrastructure: not a CPU path of the product."""
import os
import subprocess

import numpy as np
import pytest

from formation_ties.test_gpu_formation import TIE_CASES, _tied_state
from oracle.formation import FormationConfig
from oracle.lexifair import lexifair_bruteforce_batched
from test_kernel_source_host import CSRC, EMUL, ROOT, _between, _compare, _run, host_exe  # noqa: F401  (host_exe: a fixture)

_MAIN = r"""
template <int N>
static void solve(FILE* f, FILE* g, int num, int kind) {
  double c[N * N];
  int out[N];
  for (int p = 0; p < num; ++p) {
    if (fread(c, 8, N * N, f) != (size_t)(N * N)) exit(5);
    if (kind == 0) {
      if constexpr (N <= 4) fm::lexifair_small<N>(c, out); else exit(7);
    } else {
      fm::lexifair_serial<N>(c, out);
    }
    fwrite(out, 4, N, g);
  }
}
int main(int argc, char** argv) {
  if (argc != 3) return 2;
  FILE* f = fopen(argv[1], "rb"); FILE* g = fopen(argv[2], "wb");
  if (!f || !g) return 3;
  int32_t h[3];
  if (fread(h, 4, 3, f) != 3) return 4;
  switch (h[1]) {
    case 1: solve<1>(f, g, h[0], h[2]); break; case 2: solve<2>(f, g, h[0], h[2]); break;
    case 3: solve<3>(f, g, h[0], h[2]); break; case 4: solve<4>(f, g, h[0], h[2]); break;
    case 5: solve<5>(f, g, h[0], h[2]); break; case 6: solve<6>(f, g, h[0], h[2]); break;
    case 7: solve<7>(f, g, h[0], h[2]); break; case 8: solve<8>(f, g, h[0], h[2]); break;
    default: return 6;
  }
  fclose(f); fclose(g);
  return 0;
}
"""

SMALL, SERIAL = 0, 1


def cost_families(rng, num, n):
    """Cost matrices [num, n, n] per family: the ties, signed zeros, last-ulp steps and extreme magnitudes where a tie rule
    or a comparison can go wrong.  'permutation' comes with its unique answer (the other families return None)."""
    fam = {}
    fam["continuous"] = rng.random((num, n, n))
    fam["ties01"] = rng.integers(0, 2, (num, n, n)).astype(np.float64)
    fam["ties012"] = rng.integers(0, 3, (num, n, n)).astype(np.float64)
    fam["all_equal"] = np.broadcast_to(rng.random((num, 1, 1)), (num, n, n)).copy()
    fam["identical_rows"] = np.broadcast_to(rng.integers(0, 3, (num, 1, n)) * 0.25, (num, n, n)).copy()   # coincident agents
    fam["identical_cols"] = np.broadcast_to(rng.random((num, n, 1)), (num, n, n)).copy()                 # coincident goals
    fam["signed_zeros"] = np.where(rng.random((num, n, n)) < 0.3, 1.0, np.where(rng.random((num, n, n)) < 0.5, -0.0, 0.0))
    base = rng.random((num, 1, 1)) + 0.5                              # x, nextafter(x), nextafter(nextafter(x))
    up1 = np.nextafter(base, np.inf)
    fam["last_ulp"] = np.choose(rng.integers(0, 3, (num, n, n)), [base, up1, np.nextafter(up1, np.inf)])
    sub = np.finfo(np.float64).smallest_subnormal
    fam["denormals"] = rng.integers(0, 4, (num, n, n)) * sub + np.where(rng.random((num, n, n)) < 0.2, 2.0 ** -1030, 0.0)
    fam["log_uniform"] = 10.0 ** rng.uniform(-300, 300, (num, n, n))
    sigma = np.argsort(rng.random((num, n)), axis=1)                  # cost 0 on sigma, 1 elsewhere: sigma is the only answer
    perm = np.ones((num, n, n))
    np.put_along_axis(perm, sigma[..., None], 0.0, axis=2)
    fam["permutation"] = perm
    return fam, sigma


@pytest.fixture(scope="module")
def solver_exe(tmp_path_factory):
    small = open(os.path.join(CSRC, "fm_small.cuh")).read()
    form = open(os.path.join(CSRC, "fm_form.cuh")).read()
    small_body = _between(small, "// k-th permutation of 0..N-1", "}  // namespace fm")
    serial = _between(form, "template <int N>\n__device__ void lexifair_serial(", "// cdist(agent_pos, goal_pos) + lexifair")
    assert "void lexifair_small(" in small_body
    src = "\n".join(['#include "prelude.h"', "namespace fm {", small_body, serial, "}  // namespace fm", _MAIN])
    d = tmp_path_factory.mktemp("lexifair_host")
    cpp, exe = d / "lexifair_host.cpp", d / "lexifair_host"
    cpp.write_text(src)
    cmd = ["g++", "-std=c++17", "-O1", "-g", "-ffp-contract=off", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
           "-ftrivial-auto-var-init=pattern", "-I", EMUL, "-I", os.path.join(ROOT, "include"), str(cpp), "-o", str(exe)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]
    return str(exe)


def _solve(exe, tmp, costs, kind):
    num, n = costs.shape[0], costs.shape[1]
    fin, fout = os.path.join(tmp, "in.bin"), os.path.join(tmp, "out.bin")
    with open(fin, "wb") as f:
        np.array([num, n, kind], np.int32).tofile(f)
        np.ascontiguousarray(costs, dtype=np.float64).tofile(f)
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0", UBSAN_OPTIONS="print_stacktrace=1")
    res = subprocess.run([exe, fin, fout], capture_output=True, text=True, env=env)
    assert res.returncode == 0, res.stderr[-4000:]
    return np.fromfile(fout, np.int32).reshape(num, n)


def test_families_have_the_ties_they_claim():
    rng = np.random.default_rng(0)
    fam, _ = cost_families(rng, 64, 4)
    for name in ("ties01", "ties012", "all_equal", "identical_rows", "identical_cols", "signed_zeros", "last_ulp", "denormals",
                 "permutation"):
        c = fam[name].reshape(64, -1)
        assert all(np.unique(r).size < r.size for r in c), name
    z = fam["signed_zeros"]
    assert (np.signbit(z) & (z == 0)).any() and (~np.signbit(z) & (z == 0)).any()
    assert (fam["denormals"][fam["denormals"] > 0] < np.finfo(np.float64).tiny).all() and (fam["denormals"] > 0).any()
    u = fam["last_ulp"]
    assert len(np.unique(u[0])) >= 2 and np.nextafter(u[0].min(), np.inf) in u[0]


@pytest.mark.parametrize("n", range(1, 9))
def test_solvers_equal_brute_force_on_every_family(solver_exe, tmp_path, n):
    rng = np.random.default_rng(70 + n)
    num = 150 if n <= 6 else 60
    fam, sigma = cost_families(rng, num, n)
    kinds = (SMALL, SERIAL) if n <= 4 else (SERIAL,)
    for name, costs in fam.items():
        want = lexifair_bruteforce_batched(costs)
        if name == "permutation":
            assert (want == sigma).all()
        got = {k: _solve(solver_exe, str(tmp_path), costs, k) for k in kinds}
        for k, g in got.items():
            bad = np.flatnonzero((g != want).any(1))
            assert bad.size == 0, (("small", "serial")[k], name, bad[:4], costs[bad[0]], g[bad[0]], want[bad[0]])
        if n <= 4:
            assert (got[SMALL] == got[SERIAL]).all(), name


@pytest.mark.parametrize("N,O,W,fused,fair", [c for c in TIE_CASES if not c.values[2]])
def test_formation_step_source_on_tied_costs_matches_oracle(host_exe, tmp_path, N, O, W, fused, fair):  # noqa: F811
    """The tied FA / FA+FR states of formation_ties through the host build of the formation step source: goal_match bit for
    bit and every output, including the second-nearest goal of the observation, which is also decided by a tie."""
    B = 64
    cfg = FormationConfig(num_agents=N, num_obstacles=O, goal_rew=30.0, collision_rew=30.0, episode_length=25,
                          fairness_reward=fair, assignment="fair")
    st, orc = _tied_state(cfg, B, seed=10 * N + O + W)
    a = np.zeros((B, N), np.int64)
    out, post = _run(host_exe, str(tmp_path), cfg, st, actions=a, auto_reset=True)
    ref = orc.step(a, autoreset=True)
    _compare(out, ref, post, orc.get_state())
