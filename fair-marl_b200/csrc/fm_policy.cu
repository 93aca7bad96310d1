// Fused graph-network forward of the rollout policy (SURVEY.md section 8f, row N2): ONE kernel does, per graph,
//   process_adj (gnn_new.py:381-413)  ->  EmbedConv (gnn_new.py:23-141)  ->  act(TransformerConv) x (1 + gnn_layer_N)
//   (gnn_new.py:252-271, PyG TransformerConv(heads, concat=False, beta=False, edge_dim=1, root_weight=True))
//   ->  node gather (graph_aggr='node') or global mean / max / add pool (gnn_new.py:555-575)
// reading `node_obs` and `adj` exactly as the simulator's step kernel wrote them (adj once per env, shared by the N ego
// graphs of that env).  It replaces ~400 small torch kernels over [graphs, E, E, 16] edge-message tensors; the dense
// head behind it (MLPBase, GRU step, action / value layer: plain GEMMs over [graphs, 64]) stays with cuBLAS.
//
// Mapping: one WARP per graph; the weights of the network (~36 KB) live in shared memory for the whole (persistent)
// CTA, everything of a graph lives in a warp-private shared-memory scratch and in registers; no block barrier after the
// weights are loaded.  The graphs are tiny and dense (E = 2N + O + W nodes, E <= 32; ~half of the E(E-1) directed pairs
// are edges), so there is no edge list: lane (t, j) owns target node t and every LPT-th source of it (LPT = 32 / E
// lanes per target), skips the pairs that are not edges, and the LPT partial results of a target are combined with
// shuffles in a fixed order (deterministic, no atomics).
//   stage A0  hn[r]   = W_n [x_r | embed(type_r)] + b           per node      (lin1 splits into a node and an edge part)
//   stage A   x0[c]   = sum_{r -> c} LN(act(W_h LN(act(hn[r] + w_d d_rc)) + b_h))    per edge, 16-wide in registers
//   stage B1  [q|k|v|skip][n] = W_l x[n] + b_l                    dense 16 -> 160, lane = 5 output columns
//   stage B2  alpha[h,t,s] = softmax_s((q_th . k_sh + d_st (q_th . w_e,h)) / 4)      in registers, per target
//   stage B3  x'[t] = act(mean_h(sum_s alpha (v_sh + d_st w_e,h)) + skip[t])
// Supported shape family (the configuration of every shipped model_weights/*/config.yaml): embed_hidden_size =
// gnn_hidden_size = 16, gnn_num_heads = 3, gnn_concat_heads = False; any node feature width <= 17, embed_layer_N <= 2,
// any gnn_layer_N, ReLU or Tanh, with or without LayerNorm.  fp32 throughout (the parity bar is 1e-5 against the
// reference's fp32 torch modules; tests/test_gpu_policy.py).
#include <cstdio>

#include "fm_device.cuh"
#include "fm_launch.h"

namespace fm {

constexpr int GH = 16;            // embed_hidden_size == gnn_hidden_size
constexpr int GHEADS = 3;
constexpr int GHC = GHEADS * GH;  // 48
constexpr int GQW = 3 * GHC + GH; // 160 columns: q | k | v | skip
constexpr int GQS = GQW + 4;      // row stride of the q|k|v|skip scratch: 41 x 16 bytes (odd: LDS.128 conflict free over rows)
constexpr int GXS = GH + 4;       // row stride of the node-state scratch: 5 x 16 bytes
constexpr int G_WARPS = 8;

// packed weight blob (floats), see fair_marl_b200/policy.py::pack_gnn_weights
constexpr int GW_WN = 0;                       // [16 feature rows][16]  lin1 weight, node-feature part (rows >= NF-1 are zero)
constexpr int GW_TYPE = GW_WN + 16 * GH;       // [4][16]   lin1 . embed(type) + lin1 bias
constexpr int GW_WD = GW_TYPE + 4 * GH;        // [16]      lin1 weight, edge-attribute column
constexpr int GW_LN1 = GW_WD + GH;             // [16] gamma, [16] beta
constexpr int GW_EMBED_END = GW_LN1 + 2 * GH;
constexpr int GW_HID = GH * GH + GH + 2 * GH;  // per hidden embed layer: W[f][g] | b | gamma | beta
constexpr int GW_CONV = GH * GQW + GQW + GHC;  // per conv: W[k][160] | b[160] | w_e[48]

__host__ __device__ inline int gnn_weight_floats(int embed_layers, int conv_layers) {
  return GW_EMBED_END + embed_layers * GW_HID + conv_layers * GW_CONV;
}

struct GnnArgs {
  const float* w;        // packed weights
  const float* node;     // [M, E, NF]
  const float* adj;      // [M / rep, E, E]
  const int* agent_id;   // [M] node index gathered by aggr 0 (null: m % rep)
  float* out;            // [M, 16]
  int M, rep, NF, embed_layers, conv_layers, aggr, relu, ln;
  float max_edge_dist;
  int wfloats;
};

template <bool RELU>
__device__ __forceinline__ float g_act(float x) { return RELU ? fmaxf(x, 0.0f) : tanhf(x); }

// LayerNorm over 16 registers (torch: biased variance of the centred values, eps = 1e-5 inside the root)
__device__ __forceinline__ void g_layer_norm(float (&h)[GH], const float* __restrict__ gb, bool ln) {
  if (!ln) return;
  float s = 0.f;
#pragma unroll
  for (int f = 0; f < GH; ++f) s += h[f];
  const float mean = s * (1.0f / GH);
  float q = 0.f;
#pragma unroll
  for (int f = 0; f < GH; ++f) { h[f] -= mean; q = fmaf(h[f], h[f], q); }
  const float inv = rsqrtf(q * (1.0f / GH) + 1e-5f);
#pragma unroll
  for (int f = 0; f < GH; f += 4) {
    const float4 g = *reinterpret_cast<const float4*>(gb + f), b = *reinterpret_cast<const float4*>(gb + GH + f);
    h[f] = fmaf(h[f] * inv, g.x, b.x); h[f + 1] = fmaf(h[f + 1] * inv, g.y, b.y);
    h[f + 2] = fmaf(h[f + 2] * inv, g.z, b.z); h[f + 3] = fmaf(h[f + 3] * inv, g.w, b.w);
  }
}

template <int E>
struct GnnLayout {
  static constexpr int LPT = 32 / E;                          // lanes per target node
  static constexpr int SPL = (E + LPT - 1) / LPT;             // sources per lane
  static constexpr int NFP = 20;                              // padded feature row (NF <= 17)
  static constexpr int ADJ = 0, FEAT = (E * E + 3) & ~3, X = FEAT + E * NFP, Q = X + E * GXS, END = Q + E * GQS;
  static constexpr int WORDS = (END + 3) & ~3;                // floats per warp
};

// GATHER (a template parameter on the epilogue only, so that the instantiations without it keep their code): the final
// states of k = a.aggr nodes per graph side by side (agent_id [M, k] -> out [M, k * 16]).  Otherwise aggr selects one node
// (agent_id [M]) or a global pool.
template <int E, bool RELU, bool GATHER = false>
__global__ void __launch_bounds__(G_WARPS * 32, 2) gnn_kernel(const __grid_constant__ GnnArgs a) {
  using L = GnnLayout<E>;
  constexpr int LPT = L::LPT, SPL = L::SPL;
  extern __shared__ __align__(16) float smem[];
  float* W = smem;                                            // weights
  const int wpad = (a.wfloats + 3) & ~3;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  float* S = smem + wpad + wib * L::WORDS;
  for (int k = threadIdx.x; k < a.wfloats; k += blockDim.x) W[k] = __ldg(a.w + k);
  __syncthreads();
  float* s_adj = S + L::ADJ;
  float* s_feat = S + L::FEAT;
  float* s_x = S + L::X;
  float* s_q = S + L::Q;
  const bool ln = a.ln != 0;
  const int NF = a.NF, KF = NF - 1;
  // lane (t, j): target t = lane / LPT, sources s = j, j + LPT, ...
  const int t = lane / LPT, j = lane - t * LPT;
  const bool tl = t < E;                                      // this lane owns a target
  const unsigned tmask = __ballot_sync(FULL, tl);             // the lanes that do (shuffles inside `if (tl)` name only these)

  for (int m = blockIdx.x * G_WARPS + wib; m < a.M; m += gridDim.x * G_WARPS) {
    // ---- inputs -> scratch ---------------------------------------------------------------------------------
    {
      const float* ga = a.adj + (size_t)(m / a.rep) * (E * E);
      for (int k = lane; k < E * E; k += 32) s_adj[k] = __ldg(ga + k);
      const float* gn = a.node + (size_t)m * E * NF;
      for (int k = lane; k < E * NF; k += 32) { const int n = k / NF; s_feat[n * L::NFP + (k - n * NF)] = __ldcs(gn + k); }
    }
    __syncwarp();
    // ---- A0: hn[n][c] = sum_k Wn[k][c] feat[n][k] + Ttype[type_n][c]  -> s_x ------------------------------
    for (int o = lane; o < E * GH; o += 32) {
      const int n = o >> 4, c = o & 15;
      const float* f = s_feat + n * L::NFP;
      const int ty = min(max((int)f[KF], 0), 3);
      float acc = W[GW_TYPE + ty * GH + c];
      for (int k = 0; k < KF; ++k) acc = fmaf(W[GW_WN + k * GH + c], f[k], acc);
      s_x[n * GXS + c] = acc;
    }
    __syncwarp();
    // ---- A: edge messages, summed at the target -------------------------------------------------------------
    {
      float acc[GH];
#pragma unroll
      for (int f = 0; f < GH; ++f) acc[f] = 0.f;
      if (tl) {
#pragma unroll 1
        for (int r = j; r < E; r += LPT) {
          const float d = s_adj[r * E + t];                   // edge r -> t
          if (!(d < a.max_edge_dist && d > 0.0f)) continue;   // process_adj: strict <, > 0
          float h[GH];
#pragma unroll
          for (int f = 0; f < GH; f += 4) {
            const float4 hn = *reinterpret_cast<const float4*>(s_x + r * GXS + f);
            const float4 wd = *reinterpret_cast<const float4*>(W + GW_WD + f);
            h[f] = g_act<RELU>(fmaf(wd.x, d, hn.x)); h[f + 1] = g_act<RELU>(fmaf(wd.y, d, hn.y));
            h[f + 2] = g_act<RELU>(fmaf(wd.z, d, hn.z)); h[f + 3] = g_act<RELU>(fmaf(wd.w, d, hn.w));
          }
          g_layer_norm(h, W + GW_LN1, ln);
          for (int l = 0; l < a.embed_layers; ++l) {
            const float* wl = W + GW_EMBED_END + l * GW_HID;
            float o[GH];
#pragma unroll
            for (int g = 0; g < GH; g += 4) {
              const float4 b = *reinterpret_cast<const float4*>(wl + GH * GH + g);
              o[g] = b.x; o[g + 1] = b.y; o[g + 2] = b.z; o[g + 3] = b.w;
            }
#pragma unroll
            for (int f = 0; f < GH; ++f) {
#pragma unroll
              for (int g = 0; g < GH; g += 4) {
                const float4 w4 = *reinterpret_cast<const float4*>(wl + f * GH + g);   // same address in every lane: broadcast
                o[g] = fmaf(w4.x, h[f], o[g]); o[g + 1] = fmaf(w4.y, h[f], o[g + 1]);
                o[g + 2] = fmaf(w4.z, h[f], o[g + 2]); o[g + 3] = fmaf(w4.w, h[f], o[g + 3]);
              }
            }
#pragma unroll
            for (int g = 0; g < GH; ++g) h[g] = g_act<RELU>(o[g]);
            g_layer_norm(h, wl + GH * GH + GH, ln);
          }
#pragma unroll
          for (int f = 0; f < GH; ++f) acc[f] += h[f];
        }
      }
      __syncwarp();                                           // every lane has read hn before s_x is overwritten
      // the LPT partial sums of a target, in lane order
#pragma unroll
      for (int f = 0; f < GH; ++f) {
        float v = acc[f];
#pragma unroll
        for (int o = 1; o < LPT; ++o) { const float u = __shfl_down_sync(FULL, acc[f], o); if (j + o < LPT) v += u; }
        acc[f] = v;
      }
      if (tl && j == 0) {
#pragma unroll
        for (int f = 0; f < GH; f += 4) *reinterpret_cast<float4*>(s_x + t * GXS + f) = make_float4(acc[f], acc[f + 1], acc[f + 2], acc[f + 3]);
      }
    }
    __syncwarp();
    // ---- convs ----------------------------------------------------------------------------------------------
    for (int layer = 0; layer < a.conv_layers; ++layer) {
      const float* wc = W + GW_EMBED_END + a.embed_layers * GW_HID + layer * GW_CONV;
      const float* bc = wc + GH * GQW;
      const float* we = bc + GQW;
      // B1: [q | k | v | skip][n][col] for col = lane + 32 u, u < 5
      {
        constexpr int NB = E < 9 ? E : 9;                     // nodes per pass (accumulators: NB x 5)
#pragma unroll 1
        for (int n0 = 0; n0 < E; n0 += NB) {
          float acc[NB][5];
#pragma unroll
          for (int u = 0; u < 5; ++u) {
            const float b = bc[lane + 32 * u];
#pragma unroll
            for (int n = 0; n < NB; ++n) acc[n][u] = b;
          }
#pragma unroll
          for (int k0 = 0; k0 < GH; k0 += 4) {
            float w[4][5];
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
#pragma unroll
              for (int u = 0; u < 5; ++u) w[kk][u] = wc[(k0 + kk) * GQW + lane + 32 * u];
#pragma unroll
            for (int n = 0; n < NB; ++n) {
              if (n0 + n < E) {
                const float4 x4 = *reinterpret_cast<const float4*>(s_x + (n0 + n) * GXS + k0);
#pragma unroll
                for (int u = 0; u < 5; ++u) {
                  acc[n][u] = fmaf(w[0][u], x4.x, acc[n][u]); acc[n][u] = fmaf(w[1][u], x4.y, acc[n][u]);
                  acc[n][u] = fmaf(w[2][u], x4.z, acc[n][u]); acc[n][u] = fmaf(w[3][u], x4.w, acc[n][u]);
                }
              }
            }
          }
#pragma unroll
          for (int n = 0; n < NB; ++n)
            if (n0 + n < E) {
#pragma unroll
              for (int u = 0; u < 5; ++u) s_q[(n0 + n) * GQS + lane + 32 * u] = acc[n][u];
            }
        }
      }
      __syncwarp();
      // B2 + B3: attention of target t over its sources, per head, in registers
      {
        float out[GH];
#pragma unroll
        for (int c = 0; c < GH; ++c) out[c] = 0.f;
        float adsum[GHEADS] = {0.f, 0.f, 0.f};
        if (tl) {
          float sc[GHEADS][SPL], dd[SPL];
          float qe[GHEADS];
          // scores
#pragma unroll
          for (int h = 0; h < GHEADS; ++h) {
            float q[GH];
#pragma unroll
            for (int c = 0; c < GH; c += 4) {
              const float4 q4 = *reinterpret_cast<const float4*>(s_q + t * GQS + h * GH + c);
              q[c] = q4.x; q[c + 1] = q4.y; q[c + 2] = q4.z; q[c + 3] = q4.w;
            }
            float e = 0.f;
#pragma unroll
            for (int c = 0; c < GH; ++c) e = fmaf(q[c], we[h * GH + c], e);
            qe[h] = e;
#pragma unroll
            for (int i = 0; i < SPL; ++i) {
              const int s = j + i * LPT;
              float v = -INFINITY;
              if (s < E) {
                const float d = s_adj[s * E + t];             // edge s -> t
                if (h == 0) dd[i] = d;
                if (d < a.max_edge_dist && d > 0.0f) {
                  float dot = 0.f;
#pragma unroll
                  for (int c = 0; c < GH; c += 4) {
                    const float4 k4 = *reinterpret_cast<const float4*>(s_q + s * GQS + GHC + h * GH + c);
                    dot = fmaf(q[c], k4.x, dot); dot = fmaf(q[c + 1], k4.y, dot);
                    dot = fmaf(q[c + 2], k4.z, dot); dot = fmaf(q[c + 3], k4.w, dot);
                  }
                  v = (dot + qe[h] * d) * 0.25f;               // 1 / sqrt(16)
                }
              } else if (h == 0) {
                dd[i] = 0.f;
              }
              sc[h][i] = v;
            }
          }
          // softmax over the sources of (h, t): LPT lanes x SPL entries
#pragma unroll
          for (int h = 0; h < GHEADS; ++h) {
            float mx = -INFINITY;
#pragma unroll
            for (int i = 0; i < SPL; ++i) mx = fmaxf(mx, sc[h][i]);
#pragma unroll
            for (int o = 1; o < LPT; ++o) {                   // all-to-all inside the target's lane group
              const float u = __shfl_sync(tmask, mx, t * LPT + ((j + o) % LPT));
              mx = fmaxf(mx, u);
            }
            float sum = 0.f;
#pragma unroll
            for (int i = 0; i < SPL; ++i) { const float ex = sc[h][i] == -INFINITY ? 0.f : expf(sc[h][i] - mx); sc[h][i] = ex; sum += ex; }
            float tot = 0.f;                                   // fixed order: lane j = 0, 1, ... of the group
#pragma unroll
            for (int o = 0; o < LPT; ++o) tot += __shfl_sync(tmask, sum, t * LPT + o);
            const float inv = tot > 0.f ? 1.0f / tot : 0.f;   // targets without incoming edges: alpha = 0 (nan_to_num)
#pragma unroll
            for (int i = 0; i < SPL; ++i) { sc[h][i] *= inv; adsum[h] = fmaf(sc[h][i], dd[i], adsum[h]); }
          }
          // weighted values
#pragma unroll
          for (int i = 0; i < SPL; ++i) {
            const int s = j + i * LPT;
            if (s < E) {
#pragma unroll
              for (int h = 0; h < GHEADS; ++h) {
                const float al = sc[h][i];
#pragma unroll
                for (int c = 0; c < GH; c += 4) {
                  const float4 v4 = *reinterpret_cast<const float4*>(s_q + s * GQS + 2 * GHC + h * GH + c);
                  out[c] = fmaf(al, v4.x, out[c]); out[c + 1] = fmaf(al, v4.y, out[c + 1]);
                  out[c + 2] = fmaf(al, v4.z, out[c + 2]); out[c + 3] = fmaf(al, v4.w, out[c + 3]);
                }
              }
            }
          }
        }
        // combine the LPT lanes of a target (lane order), add the edge term, mean over heads, skip, activation
#pragma unroll
        for (int c = 0; c < GH; ++c) {
          float v = out[c];
#pragma unroll
          for (int o = 1; o < LPT; ++o) { const float u = __shfl_down_sync(FULL, out[c], o); if (j + o < LPT) v += u; }
          out[c] = v;
        }
#pragma unroll
        for (int h = 0; h < GHEADS; ++h) {
          float v = adsum[h];
#pragma unroll
          for (int o = 1; o < LPT; ++o) { const float u = __shfl_down_sync(FULL, adsum[h], o); if (j + o < LPT) v += u; }
          adsum[h] = v;
        }
        __syncwarp();                                         // s_x (layer input) is dead: every lane is past B1
        if (tl && j == 0) {
#pragma unroll
          for (int c = 0; c < GH; ++c) {
            float v = out[c];
#pragma unroll
            for (int h = 0; h < GHEADS; ++h) v = fmaf(adsum[h], we[h * GH + c], v);
            v = v * (1.0f / GHEADS) + s_q[t * GQS + 3 * GHC + c];
            s_x[t * GXS + c] = g_act<RELU>(v);
          }
        }
      }
      __syncwarp();
    }
    // ---- aggregation ----------------------------------------------------------------------------------------
    if constexpr (GATHER) {
      const int k = a.aggr;
      for (int o = lane; o < k * GH; o += 32) {
        const int node = a.agent_id[(size_t)m * k + (o >> 4)];
        a.out[(size_t)m * k * GH + o] = s_x[min(max(node, 0), E - 1) * GXS + (o & 15)];
      }
    } else if (lane < GH) {
      float v;
      if (a.aggr == 0) {
        const int node = a.agent_id ? a.agent_id[m] : (m % a.rep);
        v = s_x[min(max(node, 0), E - 1) * GXS + lane];
      } else {
        v = s_x[lane];
        for (int n = 1; n < E; ++n) { const float u = s_x[n * GXS + lane]; v = a.aggr == 2 ? fmaxf(v, u) : v + u; }
        if (a.aggr == 1) v *= (1.0f / E);
      }
      a.out[(size_t)m * GH + lane] = v;
    }
    __syncwarp();
  }
}

template <int E>
static cudaError_t gnn_launch_e(const GnnArgs& a, int k, cudaStream_t st) {
  using L = GnnLayout<E>;
  const size_t smem = (size_t)(((a.wfloats + 3) & ~3) + G_WARPS * L::WORDS) * sizeof(float);
  int dev = 0, sms = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return e;
  const int want = (a.M + G_WARPS - 1) / G_WARPS;
  const int grid = want < 2 * sms ? want : 2 * sms;
  if (k > 0) {                                                // multi-node gather: aggr carries k
    GnnArgs g = a;
    g.aggr = k;
    const auto kern = a.relu ? gnn_kernel<E, true, true> : gnn_kernel<E, false, true>;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, G_WARPS * 32, smem, st>>>(g);
  } else if (a.relu) {
    e = cudaFuncSetAttribute(gnn_kernel<E, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    gnn_kernel<E, true><<<grid, G_WARPS * 32, smem, st>>>(a);
  } else {
    e = cudaFuncSetAttribute(gnn_kernel<E, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    gnn_kernel<E, false><<<grid, G_WARPS * 32, smem, st>>>(a);
  }
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------------
// Second mapping of the same forward, for any 2 <= E <= 64 known only at run time: one CTA of GW_THREADS threads per graph
// (persistent over graphs), the weights in shared memory once per CTA, the graph's scratch (the warp kernel's layout,
// sized by the run-time E) after them.  A warp's scratch at E = 32 would already be 24 KB, so the warp-per-graph layout
// cannot hold these shapes; here the whole CTA works on one graph and block barriers replace __syncwarp.
//   thread (t, j), t = tid / P, j = tid % P: target t, sources j, j + P, ...  (P = GW_THREADS / EMAX adjacent lanes of one
//   warp, so a target's partial sums are still combined with shuffles in lane order);
//   stage B1: warp w projects nodes w, w + 4, w + 8, ... (lane = 5 output columns, as in the warp kernel);
//   stage B2 + B3: one head at a time, the target's scores in SPL = EMAX / P registers per thread.
// Every output element is computed by one thread in a fixed order: deterministic, and the bits of a graph do not depend on
// the CTA or the round of the persistent loop that computes it.
constexpr int GW_THREADS = 128;

__host__ __device__ inline int gnn_wide_scratch_floats(int E) {
  return ((E * E + 3) & ~3) + E * (GnnLayout<1>::NFP + GXS + GQS);
}

template <int EMAX, bool RELU, bool GATHER = false>        // GATHER: as in gnn_kernel
__global__ void __launch_bounds__(GW_THREADS, 2) gnn_wide_kernel(const __grid_constant__ GnnArgs a, const int E) {
  constexpr int P = GW_THREADS / EMAX;                        // threads per target
  constexpr int SPL = EMAX / P;                               // sources per thread (at most)
  constexpr int NFP = GnnLayout<1>::NFP;
  constexpr int NB = 8;                                       // B1: nodes per warp and pass
  constexpr int NW = GW_THREADS / 32;
  static_assert(P >= 1 && 32 % P == 0 && SPL * P == EMAX, "a target's threads must sit in one warp");
  extern __shared__ __align__(16) float smem[];
  float* W = smem;
  const int wpad = (a.wfloats + 3) & ~3;
  const int tid = threadIdx.x, lane = tid & 31, wib = tid >> 5;
  for (int k = tid; k < a.wfloats; k += GW_THREADS) W[k] = __ldg(a.w + k);
  float* s_adj = smem + wpad;
  float* s_feat = s_adj + ((E * E + 3) & ~3);
  float* s_x = s_feat + E * NFP;
  float* s_q = s_x + E * GXS;
  const bool ln = a.ln != 0;
  const int NF = a.NF, KF = NF - 1;
  const int t = tid / P, j = tid - t * P;
  const bool tl = t < E;
  const unsigned tmask = __ballot_sync(FULL, tl);
  __syncthreads();

  for (int m = blockIdx.x; m < a.M; m += gridDim.x) {
    // ---- inputs -> scratch ---------------------------------------------------------------------------------
    {
      const float* ga = a.adj + (size_t)(m / a.rep) * E * E;
      for (int k = tid; k < E * E; k += GW_THREADS) s_adj[k] = __ldg(ga + k);
      const float* gn = a.node + (size_t)m * E * NF;
      for (int k = tid; k < E * NF; k += GW_THREADS) { const int n = k / NF; s_feat[n * NFP + (k - n * NF)] = __ldcs(gn + k); }
    }
    __syncthreads();
    // ---- A0: hn[n][c] -> s_x -------------------------------------------------------------------------------
    for (int o = tid; o < E * GH; o += GW_THREADS) {
      const int n = o >> 4, c = o & 15;
      const float* f = s_feat + n * NFP;
      const int ty = min(max((int)f[KF], 0), 3);
      float acc = W[GW_TYPE + ty * GH + c];
      for (int k = 0; k < KF; ++k) acc = fmaf(W[GW_WN + k * GH + c], f[k], acc);
      s_x[n * GXS + c] = acc;
    }
    __syncthreads();
    // ---- A: edge messages, summed at the target -------------------------------------------------------------
    {
      // compensated (Kahan) sums: a thread adds up to 32 messages here, where a warp-kernel lane adds at most 19, and the
      // rounding of a long fp32 chain would otherwise grow with E
      float acc[GH], cmp[GH];
#pragma unroll
      for (int f = 0; f < GH; ++f) { acc[f] = 0.f; cmp[f] = 0.f; }
      if (tl) {
#pragma unroll 1
        for (int r = j; r < E; r += P) {
          const float d = s_adj[r * E + t];                   // edge r -> t
          if (!(d < a.max_edge_dist && d > 0.0f)) continue;   // process_adj: strict <, > 0
          float h[GH];
#pragma unroll
          for (int f = 0; f < GH; f += 4) {
            const float4 hn = *reinterpret_cast<const float4*>(s_x + r * GXS + f);
            const float4 wd = *reinterpret_cast<const float4*>(W + GW_WD + f);
            h[f] = g_act<RELU>(fmaf(wd.x, d, hn.x)); h[f + 1] = g_act<RELU>(fmaf(wd.y, d, hn.y));
            h[f + 2] = g_act<RELU>(fmaf(wd.z, d, hn.z)); h[f + 3] = g_act<RELU>(fmaf(wd.w, d, hn.w));
          }
          g_layer_norm(h, W + GW_LN1, ln);
          for (int l = 0; l < a.embed_layers; ++l) {
            const float* wl = W + GW_EMBED_END + l * GW_HID;
            float o[GH];
#pragma unroll
            for (int g = 0; g < GH; g += 4) {
              const float4 b = *reinterpret_cast<const float4*>(wl + GH * GH + g);
              o[g] = b.x; o[g + 1] = b.y; o[g + 2] = b.z; o[g + 3] = b.w;
            }
#pragma unroll
            for (int f = 0; f < GH; ++f) {
#pragma unroll
              for (int g = 0; g < GH; g += 4) {
                const float4 w4 = *reinterpret_cast<const float4*>(wl + f * GH + g);
                o[g] = fmaf(w4.x, h[f], o[g]); o[g + 1] = fmaf(w4.y, h[f], o[g + 1]);
                o[g + 2] = fmaf(w4.z, h[f], o[g + 2]); o[g + 3] = fmaf(w4.w, h[f], o[g + 3]);
              }
            }
#pragma unroll
            for (int g = 0; g < GH; ++g) h[g] = g_act<RELU>(o[g]);
            g_layer_norm(h, wl + GH * GH + GH, ln);
          }
#pragma unroll
          for (int f = 0; f < GH; ++f) {
            const float y = h[f] - cmp[f], t2 = acc[f] + y;
            cmp[f] = (t2 - acc[f]) - y;
            acc[f] = t2;
          }
        }
      }
      // the P partial sums of a target, in lane order
#pragma unroll
      for (int f = 0; f < GH; ++f) {
        float v = acc[f];
#pragma unroll
        for (int o = 1; o < P; ++o) { const float u = __shfl_down_sync(FULL, acc[f], o); if (j + o < P) v += u; }
        acc[f] = v;
      }
      __syncthreads();                                        // every thread has read hn before s_x is overwritten
      if (tl && j == 0) {
#pragma unroll
        for (int f = 0; f < GH; f += 4) *reinterpret_cast<float4*>(s_x + t * GXS + f) = make_float4(acc[f], acc[f + 1], acc[f + 2], acc[f + 3]);
      }
    }
    __syncthreads();
    // ---- convs ----------------------------------------------------------------------------------------------
    for (int layer = 0; layer < a.conv_layers; ++layer) {
      const float* wc = W + GW_EMBED_END + a.embed_layers * GW_HID + layer * GW_CONV;
      const float* bc = wc + GH * GQW;
      const float* we = bc + GQW;
      // B1: [q | k | v | skip][n][col] for col = lane + 32 u, u < 5; warp wib takes nodes wib, wib + NW, ...
      {
#pragma unroll 1
        for (int n0 = wib; n0 < E; n0 += NW * NB) {
          float acc[NB][5];
#pragma unroll
          for (int u = 0; u < 5; ++u) {
            const float b = bc[lane + 32 * u];
#pragma unroll
            for (int n = 0; n < NB; ++n) acc[n][u] = b;
          }
#pragma unroll
          for (int k0 = 0; k0 < GH; k0 += 4) {
            float w[4][5];
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
#pragma unroll
              for (int u = 0; u < 5; ++u) w[kk][u] = wc[(k0 + kk) * GQW + lane + 32 * u];
#pragma unroll
            for (int n = 0; n < NB; ++n) {
              if (n0 + n * NW < E) {
                const float4 x4 = *reinterpret_cast<const float4*>(s_x + (n0 + n * NW) * GXS + k0);
#pragma unroll
                for (int u = 0; u < 5; ++u) {
                  acc[n][u] = fmaf(w[0][u], x4.x, acc[n][u]); acc[n][u] = fmaf(w[1][u], x4.y, acc[n][u]);
                  acc[n][u] = fmaf(w[2][u], x4.z, acc[n][u]); acc[n][u] = fmaf(w[3][u], x4.w, acc[n][u]);
                }
              }
            }
          }
#pragma unroll
          for (int n = 0; n < NB; ++n)
            if (n0 + n * NW < E) {
#pragma unroll
              for (int u = 0; u < 5; ++u) s_q[(n0 + n * NW) * GQS + lane + 32 * u] = acc[n][u];
            }
        }
      }
      __syncthreads();                                        // s_q complete; s_x (the layer input) is dead from here
      // B2 + B3: attention of target t over its sources, one head at a time
      {
        float out[GH];
#pragma unroll
        for (int c = 0; c < GH; ++c) out[c] = 0.f;
        float adsum[GHEADS] = {0.f, 0.f, 0.f};
        if (tl) {
#pragma unroll
          for (int h = 0; h < GHEADS; ++h) {
            float q[GH];
#pragma unroll
            for (int c = 0; c < GH; c += 4) {
              const float4 q4 = *reinterpret_cast<const float4*>(s_q + t * GQS + h * GH + c);
              q[c] = q4.x; q[c + 1] = q4.y; q[c + 2] = q4.z; q[c + 3] = q4.w;
            }
            float qe = 0.f;
#pragma unroll
            for (int c = 0; c < GH; ++c) qe = fmaf(q[c], we[h * GH + c], qe);
            float sc[SPL];
#pragma unroll
            for (int i = 0; i < SPL; ++i) {
              const int s = j + i * P;
              float v = -INFINITY;
              if (s < E) {
                const float d = s_adj[s * E + t];             // edge s -> t
                if (d < a.max_edge_dist && d > 0.0f) {
                  float dot = 0.f;
#pragma unroll
                  for (int c = 0; c < GH; c += 4) {
                    const float4 k4 = *reinterpret_cast<const float4*>(s_q + s * GQS + GHC + h * GH + c);
                    dot = fmaf(q[c], k4.x, dot); dot = fmaf(q[c + 1], k4.y, dot);
                    dot = fmaf(q[c + 2], k4.z, dot); dot = fmaf(q[c + 3], k4.w, dot);
                  }
                  v = (dot + qe * d) * 0.25f;                 // 1 / sqrt(16)
                }
              }
              sc[i] = v;
            }
            // softmax over the sources of (h, t): P threads x SPL entries
            float mx = -INFINITY;
#pragma unroll
            for (int i = 0; i < SPL; ++i) mx = fmaxf(mx, sc[i]);
#pragma unroll
            for (int o = 1; o < P; ++o) mx = fmaxf(mx, __shfl_sync(tmask, mx, (lane & ~(P - 1)) + ((j + o) % P)));
            float sum = 0.f;
#pragma unroll
            for (int i = 0; i < SPL; ++i) { const float ex = sc[i] == -INFINITY ? 0.f : expf(sc[i] - mx); sc[i] = ex; sum += ex; }
            float tot = 0.f;                                   // fixed order: thread j = 0, 1, ... of the target
#pragma unroll
            for (int o = 0; o < P; ++o) tot += __shfl_sync(tmask, sum, (lane & ~(P - 1)) + o);
            const float inv = tot > 0.f ? 1.0f / tot : 0.f;   // targets without incoming edges: alpha = 0 (nan_to_num)
            // weighted values of this head, summed apart from the other heads' (shorter fp32 chains), compensated
            float ph[GH], pc[GH];
#pragma unroll
            for (int c = 0; c < GH; ++c) { ph[c] = 0.f; pc[c] = 0.f; }
#pragma unroll
            for (int i = 0; i < SPL; ++i) {
              const int s = j + i * P;
              if (s < E) {
                const float al = sc[i] * inv;
                adsum[h] = fmaf(al, s_adj[s * E + t], adsum[h]);
#pragma unroll
                for (int c = 0; c < GH; c += 4) {
                  const float4 v4 = *reinterpret_cast<const float4*>(s_q + s * GQS + 2 * GHC + h * GH + c);
                  const float vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
                  for (int q4 = 0; q4 < 4; ++q4) {
                    const float y = al * vv[q4] - pc[c + q4], t2 = ph[c + q4] + y;
                    pc[c + q4] = (t2 - ph[c + q4]) - y;
                    ph[c + q4] = t2;
                  }
                }
              }
            }
#pragma unroll
            for (int c = 0; c < GH; ++c) out[c] += ph[c];
          }
        }
        // combine the P threads of a target (lane order), add the edge term, mean over heads, skip, activation
#pragma unroll
        for (int c = 0; c < GH; ++c) {
          float v = out[c];
#pragma unroll
          for (int o = 1; o < P; ++o) { const float u = __shfl_down_sync(FULL, out[c], o); if (j + o < P) v += u; }
          out[c] = v;
        }
#pragma unroll
        for (int h = 0; h < GHEADS; ++h) {
          float v = adsum[h];
#pragma unroll
          for (int o = 1; o < P; ++o) { const float u = __shfl_down_sync(FULL, adsum[h], o); if (j + o < P) v += u; }
          adsum[h] = v;
        }
        if (tl && j == 0) {
#pragma unroll
          for (int c = 0; c < GH; ++c) {
            float v = out[c];
#pragma unroll
            for (int h = 0; h < GHEADS; ++h) v = fmaf(adsum[h], we[h * GH + c], v);
            v = v * (1.0f / GHEADS) + s_q[t * GQS + 3 * GHC + c];
            s_x[t * GXS + c] = g_act<RELU>(v);
          }
        }
      }
      __syncthreads();                                        // s_x complete; s_q free for the next layer
    }
    // ---- aggregation ----------------------------------------------------------------------------------------
    if constexpr (GATHER) {
      const int k = a.aggr;
      for (int o = tid; o < k * GH; o += GW_THREADS) {
        const int node = a.agent_id[(size_t)m * k + (o >> 4)];
        a.out[(size_t)m * k * GH + o] = s_x[min(max(node, 0), E - 1) * GXS + (o & 15)];
      }
    } else if (tid < GH) {
      float v;
      if (a.aggr == 0) {
        const int node = a.agent_id ? a.agent_id[m] : (m % a.rep);
        v = s_x[min(max(node, 0), E - 1) * GXS + tid];
      } else {
        v = s_x[tid];
        for (int n = 1; n < E; ++n) { const float u = s_x[n * GXS + tid]; v = a.aggr == 2 ? fmaxf(v, u) : v + u; }
        if (a.aggr == 1) v *= 1.0f / (float)E;
      }
      a.out[(size_t)m * GH + tid] = v;
    }
    __syncthreads();                                          // the scratch is read before the next graph overwrites it
  }
}

template <int EMAX, bool RELU>
static cudaError_t gnn_wide_launch_k(const GnnArgs& a, int E, int k, size_t smem, int sms, cudaStream_t st) {
  const void* kern = k > 0 ? (const void*)gnn_wide_kernel<EMAX, RELU, true> : (const void*)gnn_wide_kernel<EMAX, RELU>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  int per_sm = 0;
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, GW_THREADS, smem);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) return cudaErrorInvalidConfiguration;
  const int grid = a.M < per_sm * sms ? a.M : per_sm * sms;
  if (k > 0) {                                                // multi-node gather: aggr carries k
    GnnArgs g = a;
    g.aggr = k;
    gnn_wide_kernel<EMAX, RELU, true><<<grid, GW_THREADS, smem, st>>>(g, E);
  } else {
    gnn_wide_kernel<EMAX, RELU><<<grid, GW_THREADS, smem, st>>>(a, E);
  }
  return cudaGetLastError();
}

static cudaError_t gnn_wide_launch(const GnnArgs& a, int E, int k, cudaStream_t st) {
  const size_t smem = (size_t)(((a.wfloats + 3) & ~3) + gnn_wide_scratch_floats(E)) * sizeof(float);
  int dev = 0, sms = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return e;
  if (E <= 32) return a.relu ? gnn_wide_launch_k<32, true>(a, E, k, smem, sms, st) : gnn_wide_launch_k<32, false>(a, E, k, smem, sms, st);
  return a.relu ? gnn_wide_launch_k<64, true>(a, E, k, smem, sms, st) : gnn_wide_launch_k<64, false>(a, E, k, smem, sms, st);
}

// E values compiled: the navigation / formation shapes at N = 2..7 with O <= 3 and up to 2 walls
#define FM_GNN_CASES(X) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(17) X(19)

bool gnn_supported_entities(int E) {
#define X(e) if (E == e) return true;
  FM_GNN_CASES(X)
#undef X
  return false;
}

bool gnn_wide_supported_entities(int E) { return E >= 2 && E <= GNN_WIDE_MAX_ENTITIES; }

cudaError_t launch_gnn(const FmGnnConfig& c, const float* weights, const float* node, const float* adj, const int* agent_id,
                       float* out, int gather_k, cudaStream_t st) {
  GnnArgs a;
  a.w = weights; a.node = node; a.adj = adj; a.agent_id = agent_id; a.out = out;
  a.M = c.num_graphs; a.rep = c.graphs_per_adj; a.NF = c.node_feat_dim; a.embed_layers = c.embed_layers;
  a.conv_layers = c.conv_layers; a.aggr = c.aggr; a.relu = c.relu; a.ln = c.layer_norm;
  a.max_edge_dist = (float)c.max_edge_dist;
  a.wfloats = gnn_weight_floats(c.embed_layers, c.conv_layers);
  if (a.M <= 0) return cudaSuccess;
  const int mapping = c.mapping != 0 ? c.mapping : (gnn_supported_entities(c.num_entities) ? 1 : 2);
  if (mapping == 2) return gnn_wide_supported_entities(c.num_entities) ? gnn_wide_launch(a, c.num_entities, gather_k, st) : cudaErrorInvalidValue;
  if (mapping != 1) return cudaErrorInvalidValue;
#define X(e) if (c.num_entities == e) return gnn_launch_e<e>(a, gather_k, st);
  FM_GNN_CASES(X)
#undef X
  return cudaErrorInvalidValue;
}

int gnn_weight_count(int embed_layers, int conv_layers) { return gnn_weight_floats(embed_layers, conv_layers); }

// =====================================================================================================================
// Fused policy HEAD (everything behind the graph network): GR_Actor.forward / GR_Critic.forward after gnn_base
// (onpolicy/algorithms/graph_actor_critic.py:150-178, :380-397):
//   x = [obs | nbd]  ->  MLPBase (utils/mlp.py: LayerNorm(in), then (Linear, act, LayerNorm) x (1 + layer_N))
//     ->  RNNLayer, one step (utils/rnn.py:23-28, :57: GRU on h * mask, LayerNorm)
//     ->  actor: Categorical head (utils/act.py, distributions.py:14-28): log-softmax, mode or an inverse-CDF draw from a
//         caller-supplied uniform, log-prob of the action;   critic: v_out (a Linear; PopArt's forward is the same map).
// One WARP per row (graph); hidden_size = 64: lane l owns hidden units l and l + 32.  All weights of the head (~32 K
// floats) live in shared memory for the whole persistent CTA, stored k-quad interleaved ([k / 4][column][4]) so that one
// LDS.128 feeds four FMAs and consecutive lanes read consecutive 16-byte words; the activation vector of the row sits in
// a warp-private 64-float scratch and is read as broadcast LDS.128.  Replaces ~30 torch launches per network and step
// (LayerNorm kernels with one CTA per 64-float row, GEMVs for the 5- and 1-wide output layers, multinomial).
constexpr int HH = 64;                 // hidden_size
constexpr int HD = 32;                 // padded input width (obs_dim + 16 <= 32)
constexpr int HEAD_WARPS = 16;
constexpr int HW_FN = 0;                               // feature_norm gamma[32], beta[32]
constexpr int HW_FC1 = HW_FN + 2 * HD;                 // [8 quads][64][4], then b[64], ln gamma[64], beta[64]
constexpr int HW_FC1_SZ = HD * HH + 3 * HH;
constexpr int HW_FC_SZ = HH * HH + 3 * HH;             // per extra layer: [16 quads][64][4], b, gamma, beta
constexpr int HW_GRU_SZ = 2 * HH * 3 * HH + 2 * 3 * HH + 2 * HH;   // Wih [16][192][4] | Whh | b_ih[192] | b_hh[192] | ln gamma, beta
constexpr int HW_OUT_SZ = 8 * HH + 8;                  // Wo[8 rows][64] | bo[8]

__host__ __device__ inline int head_weight_floats(int layers, int recurrent) {
  return HW_FC1 + HW_FC1_SZ + layers * HW_FC_SZ + (recurrent ? HW_GRU_SZ : 0) + HW_OUT_SZ;
}

struct HeadArgs {
  const float* w;
  const float* obs;        // [M, obs_dim] or null (obs_dim 0)
  const float* nbd;        // [M, 16]
  const float* rnn_in;     // [M, 64]   (recurrent)
  const float* mask;       // [M]       (recurrent)
  const float* u;          // [M] uniforms in [0, 1) for the categorical draw; null: mode
  float* rnn_out;          // [M, 64]
  float* logp;             // [M]   actor
  long long* action;       // [M]   actor
  float* value;            // [M]   critic
  int M, obs_dim, layers, recurrent, feat_norm, relu, A, wfloats;
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

// LayerNorm over the 64 values held two per lane
__device__ __forceinline__ void head_ln(float& a, float& b, const float* __restrict__ g, int lane) {
  const float mean = warp_sum(a + b) * (1.0f / HH);
  a -= mean; b -= mean;
  const float var = warp_sum(fmaf(a, a, b * b)) * (1.0f / HH);
  const float inv = rsqrtf(var + 1e-5f);
  a = fmaf(a * inv, g[lane], g[HH + lane]);
  b = fmaf(b * inv, g[lane + 32], g[HH + lane + 32]);
}

// acc[c] += sum_k W[k][col_c] x[k] for NC columns of this lane; W k-quad interleaved with `ncol` columns, x in shared memory
template <int NC>
__device__ __forceinline__ void head_matvec(const float* __restrict__ Wq, int ncol, int quads, const float* __restrict__ xs,
                                            const int (&col)[NC], float (&acc)[NC]) {
#pragma unroll 4
  for (int q = 0; q < quads; ++q) {
    const float4 x4 = *reinterpret_cast<const float4*>(xs + 4 * q);
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const float4 w4 = *reinterpret_cast<const float4*>(Wq + ((size_t)q * ncol + col[c]) * 4);
      acc[c] = fmaf(w4.x, x4.x, acc[c]); acc[c] = fmaf(w4.y, x4.y, acc[c]);
      acc[c] = fmaf(w4.z, x4.z, acc[c]); acc[c] = fmaf(w4.w, x4.w, acc[c]);
    }
  }
}

template <bool RELU>
__global__ void __launch_bounds__(HEAD_WARPS * 32, 1) head_kernel(const __grid_constant__ HeadArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* W = smem;
  const int wpad = (a.wfloats + 3) & ~3;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  float* xs = smem + wpad + wib * (2 * HH);                  // activation vector | masked hidden state
  float* hs = xs + HH;
  for (int k = threadIdx.x; k < a.wfloats; k += blockDim.x) W[k] = __ldg(a.w + k);
  __syncthreads();
  const int D = a.obs_dim + GH;
  const float* w_gru = W + HW_FC1 + HW_FC1_SZ + a.layers * HW_FC_SZ;
  const float* w_out = w_gru + (a.recurrent ? HW_GRU_SZ : 0);
  const int c2[2] = {lane, lane + 32};
  for (int m = blockIdx.x * HEAD_WARPS + wib; m < a.M; m += gridDim.x * HEAD_WARPS) {
    // ---- input [obs | nbd], feature LayerNorm over D values --------------------------------------------------------
    float x = 0.f;
    if (lane < a.obs_dim) x = __ldcs(a.obs + (size_t)m * a.obs_dim + lane);
    else if (lane < D) x = __ldcs(a.nbd + (size_t)m * GH + (lane - a.obs_dim));
    if (a.feat_norm) {
      const float mean = warp_sum(x) / (float)D;
      const float d = lane < D ? x - mean : 0.f;
      const float var = warp_sum(d * d) / (float)D;
      x = lane < D ? fmaf(d * rsqrtf(var + 1e-5f), W[HW_FN + lane], W[HW_FN + HD + lane]) : 0.f;
    }
    xs[lane] = x;
    __syncwarp();
    // ---- fc1 and the layer_N hidden layers: Linear, act, LayerNorm ----------------------------------------------------
    float h0, h1;
    {
      const float* wl = W + HW_FC1;
      float acc[2] = {wl[HD * HH + lane], wl[HD * HH + lane + 32]};
      head_matvec<2>(wl, HH, HD / 4, xs, c2, acc);
      h0 = g_act<RELU>(acc[0]); h1 = g_act<RELU>(acc[1]);
      head_ln(h0, h1, wl + HD * HH + HH, lane);
    }
    __syncwarp();
    xs[lane] = h0; xs[lane + 32] = h1;
    __syncwarp();
    for (int l = 0; l < a.layers; ++l) {
      const float* wl = W + HW_FC1 + HW_FC1_SZ + l * HW_FC_SZ;
      float acc[2] = {wl[HH * HH + lane], wl[HH * HH + lane + 32]};
      head_matvec<2>(wl, HH, HH / 4, xs, c2, acc);
      h0 = g_act<RELU>(acc[0]); h1 = g_act<RELU>(acc[1]);
      head_ln(h0, h1, wl + HH * HH + HH, lane);
      __syncwarp();
      xs[lane] = h0; xs[lane + 32] = h1;
      __syncwarp();
    }
    // ---- one GRU step on h * mask (torch.nn.GRU gate order r | z | n), LayerNorm ----------------------------------------
    if (a.recurrent) {
      const float mk = a.mask[m];
      const float p0 = __ldcs(a.rnn_in + (size_t)m * HH + lane) * mk, p1 = __ldcs(a.rnn_in + (size_t)m * HH + lane + 32) * mk;
      hs[lane] = p0; hs[lane + 32] = p1;
      __syncwarp();
      const int c6[6] = {lane, lane + 32, HH + lane, HH + lane + 32, 2 * HH + lane, 2 * HH + lane + 32};
      const float* bih = w_gru + 2 * HH * 3 * HH;
      const float* bhh = bih + 3 * HH;
      float gi[6], gh[6];
#pragma unroll
      for (int c = 0; c < 6; ++c) { gi[c] = bih[c6[c]]; gh[c] = bhh[c6[c]]; }
      head_matvec<6>(w_gru, 3 * HH, HH / 4, xs, c6, gi);
      head_matvec<6>(w_gru + HH * 3 * HH, 3 * HH, HH / 4, hs, c6, gh);
      const float r0 = 1.0f / (1.0f + expf(-(gi[0] + gh[0]))), r1 = 1.0f / (1.0f + expf(-(gi[1] + gh[1])));
      const float z0 = 1.0f / (1.0f + expf(-(gi[2] + gh[2]))), z1 = 1.0f / (1.0f + expf(-(gi[3] + gh[3])));
      const float n0 = tanhf(gi[4] + r0 * gh[4]), n1 = tanhf(gi[5] + r1 * gh[5]);
      h0 = (1.0f - z0) * n0 + z0 * p0; h1 = (1.0f - z1) * n1 + z1 * p1;
      a.rnn_out[(size_t)m * HH + lane] = h0; a.rnn_out[(size_t)m * HH + lane + 32] = h1;
      head_ln(h0, h1, bhh + 3 * HH, lane);
    }
    // ---- output layer -------------------------------------------------------------------------------------------------
    float lg[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) {
      float v = 0.f;
      if (o < a.A) v = warp_sum(fmaf(w_out[o * HH + lane], h0, w_out[o * HH + lane + 32] * h1)) + w_out[8 * HH + o];
      lg[o] = v;
    }
    if (a.value) {
      if (lane == 0) a.value[m] = lg[0];
    } else {
      float mx = -INFINITY;
#pragma unroll
      for (int o = 0; o < 8; ++o) if (o < a.A) mx = fmaxf(mx, lg[o]);
      float se = 0.f;
#pragma unroll
      for (int o = 0; o < 8; ++o) if (o < a.A) se += expf(lg[o] - mx);
      const float lse = mx + logf(se);
      int act = 0;
      if (a.u) {                                             // inverse CDF of softmax(logits)
        // The fp32 sum of the probabilities can end a few ulps below 1, and u can reach 1 - 2^-24: a u at or above the
        // sum takes the last action of positive probability, never one that torch.multinomial could not draw.
        const float u = a.u[m];
        float cdf = 0.f;
        int last = 0;
        bool set = false;
#pragma unroll
        for (int o = 0; o < 8; ++o)
          if (o < a.A) {
            const float p = expf(lg[o] - lse);
            cdf += p;
            if (p > 0.f) last = o;
            if (!set && u < cdf) { act = o; set = true; }
          }
        if (!set) act = last;
      } else {                                               // FixedCategorical.mode: first maximum
        float best = -INFINITY;
#pragma unroll
        for (int o = 0; o < 8; ++o) if (o < a.A && lg[o] > best) { best = lg[o]; act = o; }
      }
      float sel = 0.f;
#pragma unroll
      for (int o = 0; o < 8; ++o) if (o == act) sel = lg[o];
      if (lane == 0) { a.action[m] = act; a.logp[m] = sel - lse; }
    }
    __syncwarp();
  }
}

int head_weight_count(int layers, int recurrent) { return head_weight_floats(layers, recurrent); }

cudaError_t launch_head(const FmHeadConfig& c, const float* weights, const float* obs, const float* nbd, const float* rnn_in,
                        const float* mask, const float* u, float* rnn_out, float* logp, long long* action, float* value,
                        cudaStream_t st) {
  HeadArgs a;
  a.w = weights; a.obs = obs; a.nbd = nbd; a.rnn_in = rnn_in; a.mask = mask; a.u = u; a.rnn_out = rnn_out; a.logp = logp;
  a.action = action; a.value = value;
  a.M = c.num_rows; a.obs_dim = c.obs_dim; a.layers = c.layers; a.recurrent = c.recurrent; a.feat_norm = c.feature_norm;
  a.relu = c.relu; a.A = c.num_outputs; a.wfloats = head_weight_floats(c.layers, c.recurrent);
  if (a.M <= 0) return cudaSuccess;
  const size_t smem = (size_t)(((a.wfloats + 3) & ~3) + HEAD_WARPS * 2 * HH) * sizeof(float);
  int dev = 0, sms = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return e;
  const int want = (a.M + HEAD_WARPS - 1) / HEAD_WARPS;
  const int grid = want < sms ? want : sms;
  if (a.relu) {
    e = cudaFuncSetAttribute(head_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    head_kernel<true><<<grid, HEAD_WARPS * 32, smem, st>>>(a);
  } else {
    e = cudaFuncSetAttribute(head_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    head_kernel<false><<<grid, HEAD_WARPS * 32, smem, st>>>(a);
  }
  return cudaGetLastError();
}

// =====================================================================================================================
// Fused CRITIC head for wide inputs: GR_Critic.forward after gnn_base (graph_actor_critic.py:323-397) on
// x = [cent_obs | nbd] of D = cent_dim + nbd_dim <= CRITIC_HEAD_MAX_IN features, where head_kernel (D <= 32) cannot serve:
// use_cent_obs (cent_obs = share_obs, the N agents' observations side by side) and critic_graph_aggr = 'node' (nbd = the
// N agent nodes' features side by side, fm_gnn_gather).  Same function as head_kernel with the value layer: feature
// LayerNorm over all D inputs -> MLPBase -> one GRU step -> v_out.
// fc1 at D = 736 is 184 KB of weights and the GRU 97.5 KB: together they do not fit a block's shared memory, so fc1 stays
// in global memory (L2) and is amortised over a tile of rows instead:
//   one WARP per tile of CH_ROWS consecutive rows (persistent); lane l owns hidden units l and l + 32, as in head_kernel;
//   the feature-LayerNorm statistics of each row over all D inputs (two passes: mean, then the centred variance);
//   fc1 over K-chunks of 32 inputs: the chunk of the tile's rows is normalised into a warp-private scratch, and each k-quad
//   of the lane's two weight columns is read once (two LDG.128) for all CH_ROWS rows;
//   everything after fc1 one row at a time, with the weights in shared memory, as head_kernel.
// The cent_obs part of a row is read from the env-level slab [M / rows_per_env, cent_dim] (row m: env m / rows_per_env).
// Every row is computed by one warp in a fixed order that does not depend on the tile it falls in: deterministic and
// batch-invariant, no atomics.
constexpr int CH_WARPS = 16;
constexpr int CH_ROWS = 8;                               // rows per warp tile
constexpr int CH_SCRATCH = CH_ROWS * HH + 2 * HH;        // per warp: fc1 chunk / fc1 outputs [CH_ROWS][64] | xs[64] | hs[64]

__host__ __device__ inline int critic_head_pad(int in_dim) { return (in_dim + 31) & ~31; }

__host__ __device__ inline int critic_head_tail_floats(int layers, int recurrent) {
  return 3 * HH + layers * HW_FC_SZ + (recurrent ? HW_GRU_SZ : 0) + HW_OUT_SZ;
}

__host__ __device__ inline int critic_head_weight_floats(int in_dim, int layers, int recurrent) {
  const int Dp = critic_head_pad(in_dim);
  return 2 * Dp + Dp * HH + critic_head_tail_floats(layers, recurrent);
}

struct CriticHeadArgs {
  const float* w;
  const float* cent;       // [M / rows_per_env, cent_dim] or null (cent_dim 0)
  const float* nbd;        // [M, nbd_dim]
  const float* rnn_in;     // [M, 64]   (recurrent)
  const float* mask;       // [M]       (recurrent)
  float* rnn_out;          // [M, 64]   (recurrent)
  float* value;            // [M]
  int M, cent_dim, rows_per_env, nbd_dim, layers, recurrent, feat_norm;
};

template <bool RELU>
__global__ void __launch_bounds__(CH_WARPS * 32, 1) critic_head_kernel(const __grid_constant__ CriticHeadArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int D = a.cent_dim + a.nbd_dim, Dp = critic_head_pad(D);
  const int tail = critic_head_tail_floats(a.layers, a.recurrent);
  float* Wfn = smem;                                         // feature_norm gamma[Dp] | beta[Dp]
  float* Wt = smem + 2 * Dp;                                 // fc1 b | ln gamma | ln beta, hidden layers, GRU, output
  const float* fc1 = a.w + 2 * Dp;                           // [Dp / 4][64][4] in global memory
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  float* xr = smem + ((2 * Dp + tail + 3) & ~3) + wib * CH_SCRATCH;
  float* xs = xr + CH_ROWS * HH;
  float* hs = xs + HH;
  for (int k = threadIdx.x; k < 2 * Dp; k += blockDim.x) Wfn[k] = __ldg(a.w + k);
  for (int k = threadIdx.x; k < tail; k += blockDim.x) Wt[k] = __ldg(fc1 + (size_t)Dp * HH + k);
  __syncthreads();
  const float* w_gru = Wt + 3 * HH + a.layers * HW_FC_SZ;
  const float* w_out = w_gru + (a.recurrent ? HW_GRU_SZ : 0);
  const int c2[2] = {lane, lane + 32};
  const int cd = a.cent_dim;
  auto in = [&](int m, int k) -> float {                    // x[m][k], k < D
    return k < cd ? __ldg(a.cent + (size_t)(m / a.rows_per_env) * cd + k) : __ldg(a.nbd + (size_t)m * a.nbd_dim + (k - cd));
  };
  const int tiles = (a.M + CH_ROWS - 1) / CH_ROWS;
  for (int tile = blockIdx.x * CH_WARPS + wib; tile < tiles; tile += gridDim.x * CH_WARPS) {
    const int m0 = tile * CH_ROWS;
    const int nr = min(CH_ROWS, a.M - m0);
    // ---- feature LayerNorm statistics over all D inputs of each row ----------------------------------------------------
    float mean[CH_ROWS], inv[CH_ROWS];
#pragma unroll
    for (int r = 0; r < CH_ROWS; ++r) {
      mean[r] = 0.f; inv[r] = 1.f;
      if (a.feat_norm && r < nr) {
        float sum = 0.f;
        for (int k = lane; k < D; k += 32) sum += in(m0 + r, k);
        const float mu = warp_sum(sum) / (float)D;
        float q = 0.f;
        for (int k = lane; k < D; k += 32) { const float d = in(m0 + r, k) - mu; q = fmaf(d, d, q); }
        mean[r] = mu;
        inv[r] = rsqrtf(warp_sum(q) / (float)D + 1e-5f);
      }
    }
    // ---- fc1 over K-chunks of 32 inputs, the weights of a chunk read once for the tile ----------------------------------
    float acc[CH_ROWS][2];
#pragma unroll
    for (int r = 0; r < CH_ROWS; ++r) { acc[r][0] = Wt[lane]; acc[r][1] = Wt[lane + 32]; }
    for (int k0 = 0; k0 < Dp; k0 += 32) {
      const int k = k0 + lane;
#pragma unroll
      for (int r = 0; r < CH_ROWS; ++r) {
        float x = 0.f;
        if (r < nr && k < D) {
          x = in(m0 + r, k);
          if (a.feat_norm) x = fmaf((x - mean[r]) * inv[r], Wfn[k], Wfn[Dp + k]);
        }
        xr[r * 32 + lane] = x;
      }
      __syncwarp();
      const float4* wq = reinterpret_cast<const float4*>(fc1 + (size_t)k0 * HH);
#pragma unroll 2
      for (int q = 0; q < 8; ++q) {
        const float4 w0 = __ldg(wq + q * HH + lane), w1 = __ldg(wq + q * HH + lane + 32);
#pragma unroll
        for (int r = 0; r < CH_ROWS; ++r) {
          const float4 x4 = *reinterpret_cast<const float4*>(xr + r * 32 + 4 * q);
          acc[r][0] = fmaf(w0.x, x4.x, acc[r][0]); acc[r][0] = fmaf(w0.y, x4.y, acc[r][0]);
          acc[r][0] = fmaf(w0.z, x4.z, acc[r][0]); acc[r][0] = fmaf(w0.w, x4.w, acc[r][0]);
          acc[r][1] = fmaf(w1.x, x4.x, acc[r][1]); acc[r][1] = fmaf(w1.y, x4.y, acc[r][1]);
          acc[r][1] = fmaf(w1.z, x4.z, acc[r][1]); acc[r][1] = fmaf(w1.w, x4.w, acc[r][1]);
        }
      }
      __syncwarp();
    }
#pragma unroll
    for (int r = 0; r < CH_ROWS; ++r) { xr[r * HH + lane] = acc[r][0]; xr[r * HH + lane + 32] = acc[r][1]; }
    __syncwarp();
    // ---- the rest of the head, one row at a time (head_kernel's arithmetic) -------------------------------------------
#pragma unroll 1
    for (int r = 0; r < nr; ++r) {
      const int m = m0 + r;
      float h0 = g_act<RELU>(xr[r * HH + lane]), h1 = g_act<RELU>(xr[r * HH + lane + 32]);
      head_ln(h0, h1, Wt + HH, lane);
      xs[lane] = h0; xs[lane + 32] = h1;
      __syncwarp();
      for (int l = 0; l < a.layers; ++l) {
        const float* wl = Wt + 3 * HH + l * HW_FC_SZ;
        float hacc[2] = {wl[HH * HH + lane], wl[HH * HH + lane + 32]};
        head_matvec<2>(wl, HH, HH / 4, xs, c2, hacc);
        h0 = g_act<RELU>(hacc[0]); h1 = g_act<RELU>(hacc[1]);
        head_ln(h0, h1, wl + HH * HH + HH, lane);
        __syncwarp();
        xs[lane] = h0; xs[lane + 32] = h1;
        __syncwarp();
      }
      if (a.recurrent) {
        const float mk = a.mask[m];
        const float p0 = __ldcs(a.rnn_in + (size_t)m * HH + lane) * mk, p1 = __ldcs(a.rnn_in + (size_t)m * HH + lane + 32) * mk;
        hs[lane] = p0; hs[lane + 32] = p1;
        __syncwarp();
        const int c6[6] = {lane, lane + 32, HH + lane, HH + lane + 32, 2 * HH + lane, 2 * HH + lane + 32};
        const float* bih = w_gru + 2 * HH * 3 * HH;
        const float* bhh = bih + 3 * HH;
        float gi[6], gh[6];
#pragma unroll
        for (int c = 0; c < 6; ++c) { gi[c] = bih[c6[c]]; gh[c] = bhh[c6[c]]; }
        head_matvec<6>(w_gru, 3 * HH, HH / 4, xs, c6, gi);
        head_matvec<6>(w_gru + HH * 3 * HH, 3 * HH, HH / 4, hs, c6, gh);
        const float r0 = 1.0f / (1.0f + expf(-(gi[0] + gh[0]))), r1 = 1.0f / (1.0f + expf(-(gi[1] + gh[1])));
        const float z0 = 1.0f / (1.0f + expf(-(gi[2] + gh[2]))), z1 = 1.0f / (1.0f + expf(-(gi[3] + gh[3])));
        const float n0 = tanhf(gi[4] + r0 * gh[4]), n1 = tanhf(gi[5] + r1 * gh[5]);
        h0 = (1.0f - z0) * n0 + z0 * p0; h1 = (1.0f - z1) * n1 + z1 * p1;
        a.rnn_out[(size_t)m * HH + lane] = h0; a.rnn_out[(size_t)m * HH + lane + 32] = h1;
        head_ln(h0, h1, bhh + 3 * HH, lane);
      }
      const float v = warp_sum(fmaf(w_out[lane], h0, w_out[lane + 32] * h1)) + w_out[8 * HH];
      if (lane == 0) a.value[m] = v;
      __syncwarp();
    }
  }
}

int critic_head_weight_count(int in_dim, int layers, int recurrent) { return critic_head_weight_floats(in_dim, layers, recurrent); }

cudaError_t launch_critic_head(const FmCriticHeadConfig& c, const float* weights, const float* cent_obs, const float* nbd,
                               const float* rnn_in, const float* mask, float* rnn_out, float* value, cudaStream_t st) {
  CriticHeadArgs a;
  a.w = weights; a.cent = cent_obs; a.nbd = nbd; a.rnn_in = rnn_in; a.mask = mask; a.rnn_out = rnn_out; a.value = value;
  a.M = c.num_rows; a.cent_dim = c.cent_dim; a.rows_per_env = c.rows_per_env; a.nbd_dim = c.nbd_dim; a.layers = c.layers;
  a.recurrent = c.recurrent; a.feat_norm = c.feature_norm;
  if (a.M <= 0) return cudaSuccess;
  const int Dp = critic_head_pad(a.cent_dim + a.nbd_dim);
  const size_t smem = (size_t)(((2 * Dp + critic_head_tail_floats(a.layers, a.recurrent) + 3) & ~3) + CH_WARPS * CH_SCRATCH) * sizeof(float);
  int dev = 0, sms = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return e;
  const int tiles = (a.M + CH_ROWS - 1) / CH_ROWS;
  const int want = (tiles + CH_WARPS - 1) / CH_WARPS;
  const int grid = want < sms ? want : sms;
  const auto kern = c.relu ? critic_head_kernel<true> : critic_head_kernel<false>;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kern<<<grid, CH_WARPS * 32, smem, st>>>(a);
  return cudaGetLastError();
}

}  // namespace fm
