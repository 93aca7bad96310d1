// Batched min-sum assignment (fm_assign_min_sum_costs / fm_assign_min_sum_positions): scipy.optimize.linear_sum_assignment
// on square problems, bit for bit.
//
// The algorithm is scipy's shortest augmenting path (rectangular_lsap.cpp after Crouse 2016; oracle/lsap.py states it),
// with its operation order and its tie rule, so that the matching equals scipy's col_ind also when several matchings tie
// for the optimum.  The per-thread form of the same loop is f_min_sum_sap (fm_form.cuh, formation OA at N >= 6).
//
// Mapping: one warp per problem.  Lane j owns column j (v, spc, path, row4col, SC and its position in `remaining`), lane i
// also owns row i (u, col4row, SR); the cost matrix sits in the warp's shared memory (8 KB at n = 32).  scipy scans
// `remaining` in order and keeps the first column of smallest spc unless a later one at the same value is unassigned; as
// one reduction that is: the smallest spc, then among columns at that value the unassigned one of LARGEST position, else
// the assigned one of SMALLEST position.  A lane therefore tracks its position in `remaining`, which changes when the
// removal of another column moves the last entry into the freed slot.  The only arithmetic is adds and subtracts, in
// scipy's order (nothing to contract).
#include <cmath>

#include "fm_device.cuh"
#include "fm_launch.h"

namespace fm {

constexpr int LSAP_WARPS = 4;

__global__ void __launch_bounds__(LSAP_WARPS * 32) lsap_kernel(const double* __restrict__ costs, const float* __restrict__ apos,
                                                               const float* __restrict__ gpos, int num, int n, int* __restrict__ out) {
  extern __shared__ __align__(16) double lsap_smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const long long prob = (long long)blockIdx.x * LSAP_WARPS + wib;
  if (prob >= num) return;                                                 // warp-uniform
  double* cost = lsap_smem + (size_t)wib * n * n;
  const int nn = n * n;
  bool finite = true;
  for (int k = lane; k < nn; k += 32) {
    double c;
    if (costs) {
      c = costs[(size_t)prob * nn + k];
    } else {
      const int i = k / n, j = k - i * n;
      const float* a = apos + ((size_t)prob * n + i) * 2;
      const float* g = gpos + ((size_t)prob * n + j) * 2;
      c = dist64(a[0], a[1], g[0], g[1]);
      finite = finite && isfinite(a[0]) && isfinite(a[1]) && isfinite(g[0]) && isfinite(g[1]);   // dist64 maps NaN to 0
    }
    finite = finite && isfinite(c);
    cost[k] = c;
  }
  if (!__all_sync(FULL, finite)) {                                         // NaN / +-inf anywhere: -1 in every entry
    if (lane < n) out[(size_t)prob * n + lane] = -1;
    return;
  }
  __syncwarp();
  double u = 0.0, v = 0.0, spc = 0.0;
  int col4row = -1, row4col = -1, path = -1;
  for (int cur = 0; cur < n; ++cur) {
    spc = INFINITY;
    bool sr = false, sc = false;
    int pos = lane < n ? n - 1 - lane : -1;                                // remaining = [n-1, n-2, ..., 0]; -1: removed
    int nrem = n, i = cur, sink = -1;
    double minv = 0.0;
    while (sink == -1) {
      if (lane == i) sr = true;
      const double ui = __shfl_sync(FULL, u, i);
      if (pos >= 0) {
        const double r = minv + cost[i * n + lane] - ui - v;
        if (r < spc) { path = i; spc = r; }
      }
      // arg-min key: (spc, tier * 32 + lane), smallest wins; tier 31 - pos (unassigned), 32 + pos (assigned), 64 (removed)
      double kv = pos >= 0 ? spc : INFINITY;
      int ks = (pos < 0 ? 64 : (row4col == -1 ? 31 - pos : 32 + pos)) * 32 + lane;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        const double ov = __shfl_xor_sync(FULL, kv, off);
        const int os = __shfl_xor_sync(FULL, ks, off);
        if (ov < kv || (ov == kv && os < ks)) { kv = ov; ks = os; }
      }
      minv = kv;
      const int j = ks & 31;
      const int rj = __shfl_sync(FULL, row4col, j);
      const int wpos = __shfl_sync(FULL, pos, j);
      if (rj == -1) sink = j; else i = rj;
      --nrem;                                                              // remaining[wpos] = remaining[--nrem]
      if (lane == j) { sc = true; pos = -1; }
      else if (pos == nrem) pos = wpos;
    }
    const double spc_own = __shfl_sync(FULL, spc, col4row < 0 ? 0 : col4row);
    if (lane == cur) u += minv;
    else if (sr) u += minv - spc_own;
    if (sc) v -= minv - spc;
    for (int j = sink;;) {                                                 // augment along path back to row cur
      const int r = __shfl_sync(FULL, path, j);
      if (lane == j) row4col = r;
      const int t = __shfl_sync(FULL, col4row, r);
      if (lane == r) col4row = j;
      j = t;
      if (r == cur) break;
    }
  }
  if (lane < n) out[(size_t)prob * n + lane] = col4row;
}

cudaError_t launch_lsap(const double* costs, const float* apos, const float* gpos, int num, int n, int* out, cudaStream_t st) {
  if (num <= 0) return cudaSuccess;
  const unsigned blocks = (unsigned)(((long long)num + LSAP_WARPS - 1) / LSAP_WARPS);
  const size_t smem = (size_t)LSAP_WARPS * n * n * sizeof(double);         // 32 KB at n = 32: below the default limit
  lsap_kernel<<<blocks, LSAP_WARPS * 32, smem, st>>>(costs, apos, gpos, num, n, out);
  return cudaGetLastError();
}

}  // namespace fm
