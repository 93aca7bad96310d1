// Training-side kernels of the device rollout buffer (fair-marl_b200/rollout.py DeviceRolloutBuffer): the returns scan of
// GraphReplayBuffer.compute_returns, the advantage normalisation of GR_MAPPO.train and the three mini-batch generators.
// fp32 on CUDA cores in the reference's operation order (every add / mul / sub / div rounded on its own: no FMA
// contraction), deterministic, no atomics, no host synchronisation.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "fm_launch.h"

namespace fm {

// value_normalizer.denormalize: x * sqrt(var) + mean, two fp32 roundings (onpolicy/utils/valuenorm.py)
static __device__ __forceinline__ float denorm(float x, const float* mean, const float* stdv) {
  return mean ? __fadd_rn(__fmul_rn(x, *stdv), *mean) : x;
}

// graph_buffer.py compute_returns, one thread per (env, agent) column walking t = T-1 .. 0.  Slab t of a [T(+1), B, N]
// field is at t * cols + col, so consecutive threads load consecutive floats.
__global__ void buffer_returns_kernel(int T, int cols, int use_gae, int proper, float g, float gl, const float* __restrict__ next_value,
                               float* __restrict__ v, const float* __restrict__ r, const float* __restrict__ m,
                               const float* __restrict__ bad, const float* __restrict__ mean, const float* __restrict__ stdv,
                               float* __restrict__ ret) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const size_t S = (size_t)cols;
  const float nv = next_value[c];
  if (use_gae) {
    v[T * S + c] = nv;                                   // value_preds[-1] = next_value
    float gae = 0.f, v1 = nv;
    for (int t = T - 1; t >= 0; --t) {
      const float v0 = v[t * S + c], m1 = m[(t + 1) * S + c];
      const float dv0 = denorm(v0, mean, stdv);
      const float delta = __fsub_rn(__fadd_rn(r[t * S + c], __fmul_rn(__fmul_rn(g, denorm(v1, mean, stdv)), m1)), dv0);
      gae = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, m1), gae));
      if (proper) gae = __fmul_rn(gae, bad[(t + 1) * S + c]);
      ret[t * S + c] = __fadd_rn(gae, dv0);
      v1 = v0;
    }
  } else {
    ret[T * S + c] = nv;                                 // returns[-1] = next_value
    float acc = nv;
    for (int t = T - 1; t >= 0; --t) {
      const float m1 = m[(t + 1) * S + c];
      acc = __fadd_rn(__fmul_rn(__fmul_rn(acc, g), m1), r[t * S + c]);
      if (proper) {
        // the reference's non-GAE branch without proper time limits does not denormalise; with them it does
        const float b1 = bad[(t + 1) * S + c];
        acc = __fadd_rn(__fmul_rn(acc, b1), __fmul_rn(__fsub_rn(1.f, b1), denorm(v[t * S + c], mean, stdv)));
      }
      ret[t * S + c] = acc;
    }
  }
}

// ---- advantages: adv = returns[:T] - denorm(value_preds[:T]); mean / population std over the active entries ----------
// Each thread keeps (count, mean, M2) by Welford's update; partials are merged by Chan's formula in a fixed tree order
// (lanes, then warps, then blocks), so the statistics are stable at any mean / std ratio and bitwise reproducible.
static constexpr int ADV_BLOCKS = 256, ADV_THREADS = 256;
static_assert(3 * ADV_BLOCKS <= FM_ADV_WORKSPACE_DOUBLES, "advantage workspace");

struct BufMoments { double n, mean, m2; };

static __device__ __forceinline__ BufMoments merge(BufMoments a, BufMoments b) {
  const double n = a.n + b.n;
  if (n == 0.0) return a;
  const double d = b.mean - a.mean, f = b.n / n;
  return {n, a.mean + d * f, a.m2 + b.m2 + d * d * a.n * f};
}

static __device__ BufMoments block_merge(BufMoments s) {
  __shared__ double sh[3][ADV_THREADS / 32];
  for (int o = 16; o > 0; o >>= 1) {
    BufMoments t{__shfl_down_sync(0xffffffffu, s.n, o), __shfl_down_sync(0xffffffffu, s.mean, o), __shfl_down_sync(0xffffffffu, s.m2, o)};
    s = merge(s, t);
  }
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { sh[0][w] = s.n; sh[1][w] = s.mean; sh[2][w] = s.m2; }
  __syncthreads();
  if (w == 0) {
    s = lane < ADV_THREADS / 32 ? BufMoments{sh[0][lane], sh[1][lane], sh[2][lane]} : BufMoments{0.0, 0.0, 0.0};
    for (int o = 16; o > 0; o >>= 1) {
      BufMoments t{__shfl_down_sync(0xffffffffu, s.n, o), __shfl_down_sync(0xffffffffu, s.mean, o), __shfl_down_sync(0xffffffffu, s.m2, o)};
      s = merge(s, t);
    }
  }
  return s;                                              // valid in thread 0
}

__global__ void __launch_bounds__(ADV_THREADS) buffer_adv_partial_kernel(long long n, const float* __restrict__ ret, const float* __restrict__ v,
                                                                 const float* __restrict__ active, const float* __restrict__ mean,
                                                                 const float* __restrict__ stdv, float* __restrict__ adv,
                                                                 double* __restrict__ part) {
  BufMoments s{0.0, 0.0, 0.0};
  for (long long i = blockIdx.x * (long long)ADV_THREADS + threadIdx.x; i < n; i += (long long)ADV_BLOCKS * ADV_THREADS) {
    const float a = __fsub_rn(ret[i], denorm(v[i], mean, stdv));
    adv[i] = a;
    if (active[i] != 0.f) {
      s.n += 1.0;
      const double x = a, d = x - s.mean;
      s.mean += d / s.n;
      s.m2 += d * (x - s.mean);
    }
  }
  s = block_merge(s);
  if (threadIdx.x == 0) {
    part[blockIdx.x] = s.n;
    part[ADV_BLOCKS + blockIdx.x] = s.mean;
    part[2 * ADV_BLOCKS + blockIdx.x] = s.m2;
  }
}

// Every block merges the ADV_BLOCKS partials in the same order (a few KB from L2), then normalises its share:
// (adv - mean) / (std + 1e-5) in fp32 as GR_MAPPO.train does with numpy float32 scalars.
__global__ void __launch_bounds__(ADV_THREADS) buffer_adv_normalise_kernel(long long n, const double* __restrict__ part, float* __restrict__ adv,
                                                                   float* __restrict__ stats) {
  __shared__ float ms[2];
  BufMoments s = threadIdx.x < ADV_BLOCKS ? BufMoments{part[threadIdx.x], part[ADV_BLOCKS + threadIdx.x], part[2 * ADV_BLOCKS + threadIdx.x]}
                                       : BufMoments{0.0, 0.0, 0.0};
  static_assert(ADV_BLOCKS == ADV_THREADS, "one partial per thread");
  s = block_merge(s);
  if (threadIdx.x == 0) {
    const float mu = s.n > 0.0 ? (float)s.mean : __int_as_float(0x7fc00000);          // nanmean of no entry: NaN
    const float sd = s.n > 0.0 ? (float)sqrt(s.m2 / s.n) : __int_as_float(0x7fc00000);
    ms[0] = mu;
    ms[1] = sd;
    if (blockIdx.x == 0) { stats[0] = mu; stats[1] = sd; }
  }
  __syncthreads();
  const float mu = ms[0], den = __fadd_rn(ms[1], 1e-5f);
  for (long long i = blockIdx.x * (long long)ADV_THREADS + threadIdx.x; i < n; i += (long long)gridDim.x * ADV_THREADS)
    adv[i] = __fdiv_rn(__fsub_rn(adv[i], mu), den);
}

// ---- mini-batch gather: one warp per output row ------------------------------------------------------------------------
struct MbArgs {
  int T, B, N, E, D, F, H;                    // H = recurrent_N * hidden_size floats per rnn state
  int mode, L, per;                           // per: samples / chunks / columns per mini-batch
  long long rows, rnn_rows, off;              // off: this mini-batch's first index into perm
  const long long* perm;
  FmBufferSlabs in;
  FmMinibatch out;
};

static __device__ __forceinline__ void copy_row(float* __restrict__ dst, const float* __restrict__ src, int n, int lane) {
  for (int i = lane; i < n; i += 32) dst[i] = __ldg(src + i);
}

__global__ void __launch_bounds__(256) buffer_minibatch_kernel(const MbArgs a) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= a.rows) return;
  int t, b, n;
  if (a.mode == FM_MINIBATCH_FEED_FORWARD) {             // flat (t, b, n): i = (t B + b) N + n
    const long long i = a.perm[a.off + row];
    n = (int)(i % a.N);
    b = (int)((i / a.N) % a.B);
    t = (int)(i / ((long long)a.N * a.B));
  } else if (a.mode == FM_MINIBATCH_RECURRENT) {         // flat (b, n, t): f = (b N + n) T + t; row l * per + c
    const long long l = row / a.per, c = row % a.per;
    const long long f = a.perm[a.off + c] * a.L + l;
    t = (int)(f % a.T);
    n = (int)((f / a.T) % a.N);
    b = (int)(f / ((long long)a.T * a.N));
  } else {                                               // naive: column j = b N + n, row t * per + c
    t = (int)(row / a.per);
    const long long j = a.perm[a.off + row % a.per];
    n = (int)(j % a.N);
    b = (int)(j / a.N);
  }
  const long long env = (long long)t * a.B + b, s = env * a.N + n;   // slab index of (t, b) and of (t, b, n)
  const int E = a.E, D = a.D, N = a.N;
  copy_row(a.out.share_obs + row * N * D, a.in.obs + env * N * D, N * D, lane);
  copy_row(a.out.obs + row * D, a.in.obs + s * D, D, lane);
  copy_row(a.out.node_obs + row * E * a.F, a.in.node_obs + s * E * a.F, E * a.F, lane);
  copy_row(a.out.adj + row * E * E, a.in.adj_env + env * E * E, E * E, lane);
  for (int i = lane; i < N; i += 32) a.out.share_agent_id[row * N + i] = i;
  if (row < a.rnn_rows) {                                // rows 0 .. rnn_rows-1 are the samples / chunk starts / t = 0 rows
    copy_row(a.out.rnn_states + row * a.H, a.in.rnn_states + s * a.H, a.H, lane);
    copy_row(a.out.rnn_states_critic + row * a.H, a.in.rnn_states_critic + s * a.H, a.H, lane);
  }
  switch (lane) {
    case 0: a.out.agent_id[row] = n; break;
    case 1: a.out.actions[row] = a.in.actions[s]; break;
    case 2: a.out.value_preds[row] = a.in.value_preds[s]; break;
    case 3: a.out.returns[row] = a.in.returns[s]; break;
    case 4: a.out.masks[row] = a.in.masks[s]; break;
    case 5: a.out.active_masks[row] = a.in.active_masks[s]; break;
    case 6: a.out.old_action_log_probs[row] = a.in.action_log_probs[s]; break;
    case 7: a.out.adv_targ[row] = a.in.advantages[s]; break;
    default: break;
  }
}

cudaError_t launch_buffer_returns(const FmReturnsConfig& c, const float* next_value, float* value_preds, const float* rewards,
                                  const float* masks, const float* bad_masks, const float* norm_mean, const float* norm_std,
                                  float* returns, cudaStream_t st) {
  const int cols = c.num_envs * c.num_agents;
  if (cols == 0) return cudaSuccess;
  buffer_returns_kernel<<<(cols + 127) / 128, 128, 0, st>>>(c.episode_length, cols, c.use_gae, c.use_proper_time_limits, c.gamma,
                                                      c.gamma_lambda, next_value, value_preds, rewards, masks, bad_masks,
                                                      norm_mean, norm_std, returns);
  return cudaGetLastError();
}

cudaError_t launch_buffer_advantages(long long n, const float* returns, const float* value_preds, const float* active_masks,
                                     const float* norm_mean, const float* norm_std, float* advantages, float* stats,
                                     double* workspace, cudaStream_t st) {
  buffer_adv_partial_kernel<<<ADV_BLOCKS, ADV_THREADS, 0, st>>>(n, returns, value_preds, active_masks, norm_mean, norm_std, advantages,
                                                         workspace);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  buffer_adv_normalise_kernel<<<ADV_BLOCKS, ADV_THREADS, 0, st>>>(n, workspace, advantages, stats);
  return cudaGetLastError();
}

cudaError_t launch_buffer_minibatch(const FmMinibatchConfig& c, long long rows, long long rnn_rows, int per, long long off,
                                    const FmBufferSlabs& in, const long long* perm, const FmMinibatch& out, cudaStream_t st) {
  if (rows == 0) return cudaSuccess;
  MbArgs a{c.episode_length, c.num_envs, c.num_agents, c.num_entities, c.obs_dim, c.node_feat_dim, c.rnn_floats,
           c.mode, c.data_chunk_length, per, rows, rnn_rows, off, perm, in, out};
  buffer_minibatch_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(a);
  return cudaGetLastError();
}

}  // namespace fm
