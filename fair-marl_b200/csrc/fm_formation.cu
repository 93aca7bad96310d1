// Formation-family scenarios on the device (SURVEY.md section 8f, row N3).
//
// Reference: multiagent/custom_scenarios/nav_fairassign_fairrew_formation_graph.py (FA+FR), its twin
// nav_fairassign_nofairrew_formation_graph.py (FA), and the base scenarios nav_base_formation_graph_mask.py (OA: the reward
// distance is the agent's entry of the min-sum matching re-solved in agent 0's reward call, :666-706) and
// nav_base_formation_graph_randomgoal.py (RA: a random permutation drawn at reset, :258-259), driven by
// MultiAgentGraphEnv.step (environment.py:816-877) over World.step (core.py:250-404).  oracle/formation.py is the float64
// restatement these kernels are tested against (pinned to 1 733 steps of the unmodified reference).
//
// Mapping.  The per-agent loop of MultiAgentGraphEnv.step is inherently sequential in this family (agent i's observation
// rewrites the goal-occupancy table agent i + 1 reads, agent 0's reward call re-solves the assignment, a latching agent's
// velocity is zeroed between its observation and its node rows), so the LOGIC runs one thread per env, lanes of a warp =
// 32 consecutive envs, walking the reference's own order with the env in registers / local memory (float64 like the
// reference, except the softplus contact terms, which are the fp32 hardware-approximation form of the navigation
// kernels).  What a thread produces is not the output rows but their RECIPE, in warp-private shared memory:
//   obs / reward / done   lane = env images in API layout (the warp's slice of each array is one contiguous range)
//   adj, node_obs         fp32 positions + post-integration velocities + per agent the ego index from which its velocity
//                         reads zero (it latched this step) + per (ego, agent) the goal it is shown heading for (landmark
//                         index, occupied, history): 2 E + 3 N + 3 N^2 floats per env (55 at N = 3, O = 3)
// and the EMISSION is warp-cooperative: the images go out as TMA bulk stores; adj (unique pairs spread over the lanes,
// mirrored) and the 13-float node rows are rebuilt from the recipes into two small staging buffers, one being filled
// while the copy engine streams the other.  14.7 KB of shared memory per warp at N = 3: 14 warps / SM -- the logic is a
// latency-bound serial chain, so resident warps are what buys throughput (round 2, first version: whole-tile adj image +
// 6 N^2-float recipes, 29.9 KB, 7 warps / SM, 20 % of the HBM roofline; round 1: 468-byte row runs per lane, 8.5 %).
//
// The device functions below are also compiled for the host by tests/test_kernel_source_host.py (g++, ASan + UBSan,
// tests/host_emul/prelude.h stands in for the CUDA built-ins): the per-env logic and the row builder are checked against
// the oracle on the CPU; only the warp-level emission (form_emit) is GPU-only.
#include "fm_form.cuh"

namespace fm {

// ===================================================================================================================
// Device only from here: shared-memory tile of a warp, warp-cooperative emission, kernels, launcher.
#ifdef __CUDACC__

// The warp's images -> global memory.  Full, 16-byte aligned tiles go through the copy engine (obs / reward / done images
// as they are; adj and the node rows rebuilt from the recipes into two staging buffers, one being filled while the engine
// streams the other); ragged / unaligned tiles are written by the lanes.
template <int N>
__device__ void form_emit(const FormParams& p, float* __restrict__ S, const FormTile& t, int env0, int nenv, int lane, bool with_step) {
  const int O = p.O, W = p.W, E = 2 * N + O + W, NE = N * E, EE = E * E, wall_hist = p.assignment == 0;
  float* g_obs = p.out.obs ? p.out.obs + (size_t)env0 * N * F_OBS : nullptr;
  float* g_adj = p.out.adj ? p.out.adj + (size_t)env0 * EE : nullptr;
  float* g_rew = (with_step && p.out.reward) ? p.out.reward + (size_t)env0 * N : nullptr;
  uint8_t* g_done = (with_step && p.out.done) ? p.out.done + (size_t)env0 * N : nullptr;
  float* g_node = p.out.node_obs ? p.out.node_obs + (size_t)env0 * NE * F_NODE : nullptr;
  const bool bulk = nenv == 32 && aligned16(g_obs) && aligned16(g_adj) && aligned16(g_rew) && aligned16(g_done) && aligned16(g_node);
  const float* rec = S + t.rec;
  if (!bulk) {
    if (g_obs) for (int k = lane; k < nenv * N * F_OBS; k += 32) __stcs(g_obs + k, S[t.obs + k]);
    if (g_rew) for (int k = lane; k < nenv * N; k += 32) __stcs(g_rew + k, S[t.rew + k]);
    if (g_done) for (int k = lane; k < nenv * N; k += 32) g_done[k] = reinterpret_cast<const uint8_t*>(S + t.done)[k];
    if (g_adj)
      for (int k = lane; k < nenv * EE; k += 32) {
        const int el = k / EE, q = k - el * EE, a = q / E;
        __stcs(g_adj + k, f_adj_elem(rec + el * t.rec_stride, a, q - a * E));
      }
    if (g_node)
      for (int r = lane; r < nenv * NE; r += 32) {
        const int el = r / NE, q = r - el * NE, i = q / E;
        float row[F_NODE];
        f_row(rec + el * t.rec_stride, N, O, i, q - i * E, row, W, wall_hist);
#pragma unroll
        for (int f = 0; f < F_NODE; ++f) __stcs(g_node + (size_t)r * F_NODE + f, row[f]);
      }
    return;
  }
  uint64_t pol = 0;
  if (lane == 0) {
    pol = evict_first_policy();
    fence_async_smem();
    if (g_obs) bulk_store(g_obs, S + t.obs, 32 * N * F_OBS * 4, pol);
    if (g_rew) bulk_store(g_rew, S + t.rew, 32 * N * 4, pol);
    if (g_done) bulk_store(g_done, S + t.done, 32 * N, pol);
    bulk_commit();
  }
  int c = 0;                                                                // staging chunks issued so far
  auto next_buffer = [&]() -> float* {
    if (c >= 2) { if (lane == 0) bulk_wait_read<1>(); __syncwarp(); }       // the engine has read chunk c - 2 out of this buffer
    return S + t.stage + (c & 1) * F_CHUNK_WORDS;
  };
  auto send = [&](float* gdst, const float* buf, int words) {
    __syncwarp();
    if (lane == 0) { fence_async_smem(); bulk_store(gdst, buf, (uint32_t)words * 4u, pol); bulk_commit(); }
    ++c;
  };
  if (g_adj) {
    // k whole envs per chunk (k a multiple of 4: 16-byte sizes): the unique pairs a < c of each env are spread over the
    // lanes and mirrored; k = 0 (E >= 15): element-wise, straight to global memory (coalesced)
    const int k = (E * (E - 1) / 2 > 96) ? 0 : (8 * EE <= F_CHUNK_WORDS ? 8 : (4 * EE <= F_CHUNK_WORDS ? 4 : 0));
    if (k == 0) {
      for (int q = lane; q < 32 * EE; q += 32) {
        const int el = q / EE, w = q - el * EE, a = w / E;
        __stcs(g_adj + q, f_adj_elem(rec + el * t.rec_stride, a, w - a * E));
      }
    } else {
      // pair w -> (a, c), a < c, decoded once per launch into the lane's registers (P <= 3 x 32 for the E that get here)
      const int P = E * (E - 1) / 2;
      int pa[3], pc[3];
#pragma unroll
      for (int u = 0; u < 3; ++u) {
        int w = lane + 32 * u, a = 0;
        if (w < P) { while (w >= E - 1 - a) { w -= E - 1 - a; ++a; } }
        pa[u] = a; pc[u] = a + 1 + w;
      }
      for (int e0 = 0; e0 < 32; e0 += k) {
        float* buf = next_buffer();
        for (int el = 0; el < k; ++el) {
          const float* r = rec + (e0 + el) * t.rec_stride;
          float* img = buf + el * EE;
          if (lane < E) img[lane * E + lane] = 0.0f;
#pragma unroll
          for (int u = 0; u < 3; ++u)
            if (lane + 32 * u < P) {
              const float d = f_adj_elem(r, pa[u], pc[u]);
              img[pa[u] * E + pc[u]] = d; img[pc[u] * E + pa[u]] = d;
            }
        }
        send(g_adj + (size_t)e0 * EE, buf, k * EE);
      }
    }
  }
  if (g_node) {
    const int rows = 32 * NE;                                               // a multiple of 4 rows: 16-byte chunk sizes
    // row r of the warp = (env el, ego i, entity en); the lane's row advances by one chunk per iteration: carried, not divided
    static_assert(F_ROWS_PER_LANE == 1, "one row per lane and chunk");
    const int adv_i = F_CHUNK_ROWS / E, adv_e = F_CHUNK_ROWS - adv_i * E;
    int el = lane / NE, i = (lane - el * NE) / E, en = lane - el * NE - i * E;
    for (int r0 = 0; r0 < rows; r0 += F_CHUNK_ROWS) {
      float* buf = next_buffer();
      if (r0 + lane < rows) f_row(rec + el * t.rec_stride, N, O, i, en, buf + lane * F_NODE, W, wall_hist);
      en += adv_e; i += adv_i;
      if (en >= E) { en -= E; ++i; }
      while (i >= N) { i -= N; ++el; }
      send(g_node + (size_t)r0 * F_NODE, buf, min(F_CHUNK_ROWS, rows - r0) * F_NODE);
    }
  }
  if (lane == 0) bulk_wait_read<0>();
}

// Episode statistics of one step into the warp's own row of p.stats (layout of fm_stats_read): per agent the emitted reward,
// per agent the 14 info values of the envs whose agents are all done, the number of those envs and the env-steps.  Lane =
// env; reward and done come from the warp's images, info from the row this lane has just written.  Lanes >= nenv add 0.
// Only lane 0 adds into the row and only this warp owns it, so the order of the adds is fixed: the sums are deterministic
// (reductions from one thread to one address are performed in program order).
// A global-space reduction: fire-and-forget.  Through the generic atomicAdd(double*) the compiler emits a returning ATOM
// behind a shared-memory CAS-loop branch here (it cannot see that p.stats is global), and lane 0 waits for every result.
__device__ __forceinline__ void red_add(double* a, double v) {
  asm volatile("red.global.add.f64 [%0], %1;" :: "l"(__cvta_generic_to_global(a)), "d"(v) : "memory");
}

template <int N>
__device__ __forceinline__ void form_stats(const FormParams& p, const float* S, const FormTile& t, int env0, int nenv, int lane) {
  double* row = p.stats + (size_t)(env0 >> 5) * (15 * N + 2);
  const bool live = lane < nenv;
  const uint8_t* done = reinterpret_cast<const uint8_t*>(S + t.done) + lane * N;
  bool all_done = live;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    double r = live ? (double)S[t.rew + lane * N + i] : 0.0;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) r += __shfl_xor_sync(FULL, r, off);
    if (lane == 0) red_add(row + i, r);
    all_done = all_done && done[i] == 1;
  }
  if (__any_sync(FULL, all_done)) {
    const float* info = p.out.info + (size_t)(env0 + (live ? lane : 0)) * N * INFO_F;
#pragma unroll 1
    for (int q = 0; q < N * INFO_F; ++q) {
      double v = all_done ? (double)info[q] : 0.0;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(FULL, v, off);
      if (lane == 0) red_add(row + N + q, v);
    }
  }
  const unsigned term = __ballot_sync(FULL, all_done);
  if (lane == 0) { red_add(row + 15 * N, (double)__popc(term)); red_add(row + 15 * N + 1, (double)nenv); }
}

constexpr int FORM_WARPS = 1;          // no block-level cooperation: one warp per CTA packs the SM's shared memory best
#ifndef FM_FORM_MIN_BLOCKS
#define FM_FORM_MIN_BLOCKS 1           // A/B knob (FM_NVCC_EXTRA=-DFM_FORM_MIN_BLOCKS=n): resident warps ptxas must leave room for
#endif

template <int N, int MODE, int OT>
__global__ void __launch_bounds__(FORM_WARPS * 32, FM_FORM_MIN_BLOCKS) formation_kernel(const FormParams p) {
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int env0 = (blockIdx.x * FORM_WARPS + wib) * 32;
  if (env0 >= p.B) return;                                                  // warp-uniform
  const int nenv = min(32, p.B - env0);
  const FormTile t = form_tile(N, p.O, p.W);
  float* S = smem + (size_t)wib * t.words;
  if (lane < nenv) {
    FOut o;
    o.obs = S + t.obs + lane * N * F_OBS; o.rew = S + t.rew + lane * N;
    o.done = reinterpret_cast<uint8_t*>(S + t.done) + lane * N; o.rec = S + t.rec + lane * t.rec_stride;
    if (MODE == 0) form_step_env<N, OT>(p, env0 + lane, o); else form_reset_env<N>(p, env0 + lane, o);
  }
  __syncwarp();
  if (MODE == 0 && p.stats) form_stats<N>(p, S, t, env0, nenv, lane);
  form_emit<N>(p, S, t, env0, nenv, lane, MODE == 0);
}

int formation_max_agents() { return 7; }

// ---- split path of the small teams (N <= 4, O <= 3): LOGIC kernel + IMAGE kernel --------------------------------------
// The per-env logic is one long dependent chain per thread (about 6 000 warp instructions per 32 envs, float64), and 65 536
// envs are only 2 048 warps: one wave in which every warp walks that chain at one instruction per ~13 cycles.  Rebuilding
// adj and the node rows from the recipes doubled the chain when the same warp did it afterwards (round 2, profiles/
// r02_e / r02_f: 26 M warp instructions, half of them emission, issue slots 35 % busy).  So the step is two launches:
//   formation_logic_kernel   thread per env, env in registers; obs / reward / done images and the 32 recipes of the tile
//                            leave through TMA bulk stores (the recipes into a handle-owned block, tile-contiguous)
//   formation_image_kernel   four warps per tile, lane = env: the rows (ego i, entity en) and the unique adj pairs are
//                            spread over the warps with warp-uniform (i, en) / (a, c), written into shared-memory IMAGES of
//                            the API layout (odd env strides at N = 3: conflict free) and handed to the copy engine as two
//                            bulk stores per tile.  No long chain, 12 warps per SM in flight, bound by the stores.
#ifndef FM_FORM_LOGIC_BLOCKS
#define FM_FORM_LOGIC_BLOCKS 16        // 128 registers: measured 74 us against 85 (168 registers) and 85 (239, no cap) at C2 shape
#endif
template <int N, int OT>
__global__ void __launch_bounds__(32, FM_FORM_LOGIC_BLOCKS) formation_logic_kernel(const FormParams p) {
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x;
  const int env0 = blockIdx.x * 32;
  const int nenv = min(32, p.B - env0);
  // The image kernel is a programmatic dependent launch: it may be scheduled as soon as every CTA of this grid is running,
  // and each of its CTAs waits for the `ready` flag of its own 16 envs.  So rows are built while the few warps in which an
  // env finished early are still walking the serial reset + re-observation (which set this kernel's duration: 29 us on the
  // steps without an early reset, 55 with one -- same instruction total, profiles/r02_n, tools/form_tail_probe.py).
  if (p.ready) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const FormTile t = form_tile(N, OT, 0, false);
  float* S = smem;
  if (lane < nenv) {
    FOut o;
    o.obs = S + t.obs + lane * N * F_OBS; o.rew = S + t.rew + lane * N;
    o.done = reinterpret_cast<uint8_t*>(S + t.done) + lane * N; o.rec = S + t.rec + lane * t.rec_stride;
    form_step_env<N, OT>(p, env0 + lane, o);
  }
  __syncwarp();
  if (p.stats) form_stats<N>(p, S, t, env0, nenv, lane);
  float* g_obs = p.out.obs ? p.out.obs + (size_t)env0 * N * F_OBS : nullptr;
  float* g_rew = p.out.reward ? p.out.reward + (size_t)env0 * N : nullptr;
  uint8_t* g_done = p.out.done ? p.out.done + (size_t)env0 * N : nullptr;
  float* g_rec = p.rec + (size_t)blockIdx.x * 32 * t.rec_stride;           // handle-owned, whole tiles, 128-byte multiples
  const bool bulk = nenv == 32 && aligned16(g_obs) && aligned16(g_rew) && aligned16(g_done);
  if (p.ready) {
    // recipes by plain coalesced stores, then fence + flags: the consumer's acquire load orders its reads behind them
    for (int k = lane; k < 32 * t.rec_stride; k += 32) g_rec[k] = S[t.rec + k];
    __threadfence();
    __syncwarp();
    if (lane < 2) {
      int* f = p.ready + 2 * blockIdx.x + lane;
      asm volatile("st.release.gpu.global.s32 [%0], %1;" :: "l"(f), "r"(1) : "memory");
    }
  }
  if (lane == 0) {
    const uint64_t pol = evict_first_policy();
    fence_async_smem();
    if (!p.ready) bulk_store_plain(g_rec, S + t.rec, 32u * (uint32_t)t.rec_stride * 4u);  // read back by the image kernel: default L2 policy
    if (bulk) {
      if (g_obs) bulk_store(g_obs, S + t.obs, 32 * N * F_OBS * 4, pol);
      if (g_rew) bulk_store(g_rew, S + t.rew, 32 * N * 4, pol);
      if (g_done) bulk_store(g_done, S + t.done, 32 * N, pol);
    }
    bulk_commit();
  }
  if (!bulk) {
    if (g_obs) for (int k = lane; k < nenv * N * F_OBS; k += 32) __stcs(g_obs + k, S[t.obs + k]);
    if (g_rew) for (int k = lane; k < nenv * N; k += 32) __stcs(g_rew + k, S[t.rew + k]);
    if (g_done) for (int k = lane; k < nenv * N; k += 32) g_done[k] = reinterpret_cast<const uint8_t*>(S + t.done)[k];
  }
  if (lane == 0) bulk_wait_read<0>();
}

template <int N, int OT>
static cudaError_t launch_formation_split(const FormParams& p, cudaStream_t st, const FormAsync* async) {
  const FormTile t = form_tile(N, OT, 0, false);
  const size_t smem = (size_t)t.words * sizeof(float);
  static int attr_device = -1;                         // opt-in shared-memory size: once per device
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev != attr_device) {
    e = cudaFuncSetAttribute(formation_logic_kernel<N, OT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    // 65 536 envs are 2 048 one-warp CTAs and 148 SMs x 14 resident CTAs is 2 072: with the carve-out the driver picked by
    // itself some launches fitted one wave (27 us) and most did not (55 us; same instructions, profiles/r02_l).  Ask for
    // the largest shared-memory carve-out so that the register file (16 CTAs / SM) is the only limit.
    e = cudaFuncSetAttribute(formation_logic_kernel<N, OT>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    attr_device = dev;
  }
  // Pending resets: the envs that reset in EARLIER steps consumed their blocks; redraw them on the side stream while this
  // step runs (forked before the logic launch, so that logic -> image stay adjacent for the dependent launch; joined behind
  // the image kernel).  A block is therefore fresh again two steps after it was used; an env that resets sooner draws inline.
  const bool pf = async && p.pend && p.auto_reset;
  if (pf) {
    if ((e = cudaEventRecord(async->fork, st)) != cudaSuccess) return e;
    if ((e = cudaStreamWaitEvent(async->side, async->fork, 0)) != cudaSuccess) return e;
    if ((e = launch_formation_prefetch(p, async->side)) != cudaSuccess) return e;
    if ((e = cudaEventRecord(async->join, async->side)) != cudaSuccess) return e;
  }
  const bool images = p.out.node_obs || p.out.adj;
  FormParams lp = p;
  if (!images) lp.ready = nullptr;                    // no image kernel behind this step: nobody would consume (and clear) the flags
  formation_logic_kernel<N, OT><<<(p.B + 31) / 32, 32, smem, st>>>(lp);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if (images)
    if ((e = launch_formation_image(p, st)) != cudaSuccess) return e;                // fm_form_image.cu
  if (pf) e = cudaStreamWaitEvent(st, async->join, 0);
  return e;
}

template <int N, int MODE, int OT>
static cudaError_t launch_formation_k(const FormParams& p, cudaStream_t st) {
  const FormTile t = form_tile(N, p.O, p.W);
  const size_t smem = (size_t)t.words * FORM_WARPS * sizeof(float);
  const int blocks = (p.B + 32 * FORM_WARPS - 1) / (32 * FORM_WARPS);
  cudaError_t e = cudaFuncSetAttribute(formation_kernel<N, MODE, OT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  formation_kernel<N, MODE, OT><<<blocks, FORM_WARPS * 32, smem, st>>>(p);
  return cudaGetLastError();
}

// Steps of small teams (N <= 4) with at most 3 obstacles take the split path (env in registers, obstacle count a template
// parameter, image kernel); everything else, and every reset, the fused generic kernel.
template <int N>
static cudaError_t launch_formation_n(const FormParams& p, bool is_reset, cudaStream_t st, const FormAsync* async) {
  if (is_reset) return launch_formation_k<N, 1, -1>(p, st);
  if constexpr (N <= 4) {
    if (p.rec && !p.fused && p.W == 0) {
      switch (p.O) {
        case 0: return launch_formation_split<N, 0>(p, st, async);
        case 1: return launch_formation_split<N, 1>(p, st, async);
        case 2: return launch_formation_split<N, 2>(p, st, async);
        case 3: return launch_formation_split<N, 3>(p, st, async);
        default: break;
      }
    }
  }
  return launch_formation_k<N, 0, -1>(p, st);
}

size_t formation_pending_floats(int N, int O, int B) { return (size_t)form_pending_floats(N, O) * (size_t)(((B + 31) / 32) * 32); }
size_t formation_recipe_floats(int N, int O, int B) { return (size_t)((B + 31) / 32) * 32 * form_tile(N, O).rec_stride; }

cudaError_t launch_formation(const FormParams& p, bool is_reset, cudaStream_t st, const FormAsync* async) {
  switch (p.N) {
    case 2: return launch_formation_n<2>(p, is_reset, st, async);
    case 3: return launch_formation_n<3>(p, is_reset, st, async);
    case 4: return launch_formation_n<4>(p, is_reset, st, async);
    case 5: return launch_formation_n<5>(p, is_reset, st, async);
    case 6: return launch_formation_n<6>(p, is_reset, st, async);
    case 7: return launch_formation_n<7>(p, is_reset, st, async);
    default: return cudaErrorInvalidValue;
  }
}

#endif  // __CUDACC__

}  // namespace fm
