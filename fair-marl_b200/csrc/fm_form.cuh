// Formation family: per-env device functions shared by the kernels of fm_formation.cu (fused and logic kernels) and
// fm_form_image.cu (image kernel), and compiled for the host by tests/test_kernel_source_host.py.
#pragma once
#include "fm_device.cuh"
#include "fm_launch.h"
#include "fm_small.cuh"

#ifndef FM_SQRT64
#define FM_SQRT64 dsqrt_fast      // correctly rounded, branch free (fm_device.cuh); the host build uses sqrt
#endif
#ifndef FM_DIV64
#define FM_DIV64 ddiv_fast        // a / b for normal b > 0, branch free, relative error ~1e-16 (fm_device.cuh): the quotients
#endif                            // here end in float32 outputs / state; the host build divides

namespace fm {

constexpr int F_OBS = FM_FORMATION_OBS_DIM, F_NODE = FM_FORMATION_NODE_FEAT_DIM, F_MAXO = FM_FORMATION_MAX_OBSTACLES;
constexpr int F_ROWS_PER_LANE = 1, F_CHUNK_ROWS = 32 * F_ROWS_PER_LANE, F_CHUNK_WORDS = F_CHUNK_ROWS * F_NODE;   // 32 rows, 416 floats (small: shared memory per warp bounds the occupancy)

// Unrolling policy.  For N <= 4 every loop over agents / goals is fully unrolled so that the env (FEnv) is scalarised into
// registers: with runtime indices it lives in local memory, 0.9 KB per thread, far more than the L1 left beside the shared
// memory of 14 warps -- the round-2 profile of the first version showed 36 % of the stalls on those L2 round trips.
// Runtime indices (the goal an agent is matched to, the chosen goal of an observation) go through ld / st / ldm below:
// select chains for N <= 4, plain indexing for larger teams (which keep the env in local memory).  OT >= 0 is the
// compile-time obstacle count of the specialised instantiations, -1 reads p.O.
#define FM_UNROLL_N _Pragma("unroll (N <= 4 ? 16 : 1)")
#define FM_UNROLL_O _Pragma("unroll (OT >= 0 ? 8 : 1)")

template <int L, typename T>
__device__ __forceinline__ T ld(const T (&a)[L], int k) {
  if constexpr (L <= 4) {
    T r = a[0];
#pragma unroll
    for (int j = 1; j < L; ++j) r = (k == j) ? a[j] : r;
    return r;
  } else {
    return a[k];
  }
}
template <int L, typename T, typename V>
__device__ __forceinline__ void st(T (&a)[L], int k, V v) {
  if constexpr (L <= 4) {
#pragma unroll
    for (int j = 0; j < L; ++j) a[j] = (k == j) ? (T)v : a[j];
  } else {
    a[k] = (T)v;
  }
}
// m[r][c] of an N x N matrix: r is a compile-time value after unrolling, c a runtime index
template <int N>
__device__ __forceinline__ double ldm(const double (&m)[N * N], int r, int c) {
  if constexpr (N <= 4) {
    double v = m[r * N];
#pragma unroll
    for (int j = 1; j < N; ++j) v = (c == j) ? m[r * N + j] : v;
    return v;
  } else {
    return m[r * N + c];
  }
}

// One env in a thread.  Positions, velocities and the running statistics are float64 (the step computes in float64 like
// the reference); what is only ever a float32 value, a small integer or an index keeps its storage type (static entity
// positions, goal history, nearest-landmark latch, collision counters, min_time): the conversions are exact.
template <int N>
struct FEnv {
  double px[N], py[N], vx[N], vy[N], pd[N];
  float lx[N], ly[N], ox[F_MAXO], oy[F_MAXO];
  float wax[2], wlen;          // walls (0..2): axis position per wall, half-length per env (:233-234, :301-333)
  int wor[2];                  // orientation per wall: 0 'H' (along x at y = axis), 1 'V'
  double occ[N], dtg[N], treq[N], dleft[N];
  float hist[N], reached[N], mint[N], nac[N], noc[N];
  int gm[N];
  bool status[N];
  double dmean, dstd;
  int step, episode;
  // agent a -> landmark g distances at the current positions (f_dists): positions do not move inside the per-agent loop of
  // a step, and observation, reward, node rows, info and the assignment all read this same matrix (the reference
  // recomputes each entry up to N + 4 times per step)
  double dal[N * N];
};

// Where one env's thread writes (shared memory on the device, lane = env; plain arrays in the host harness).
struct FOut {
  float* obs;      // [N][11]
  float* rew;      // [N]
  uint8_t* done;   // [N]
  float* rec;      // recipe of adj and the node rows:
                   //   pos [E][2] | vel [N][2] after the integration | latch [N]: ego index from which agent a's velocity reads 0
                   //   (it latched in this step's reward call of that ego; N + 1: never) | per ego i: pick [N][3] = (goal: landmark
                   //   index, or -1 = the agent's own position; goal occupied; goal history) as shown in ego i's rows
};
// with walls: their midpoints close the position list (E = 2 N + O + W), and (half-length, axis 0, axis 1) follow the picks
__host__ __device__ inline int form_rec_floats(int N, int O, int W = 0) { return 2 * (2 * N + O + W) + 3 * N + 3 * N * N + (W ? 3 : 0); }

__device__ __forceinline__ double dn(double dx, double dy) {      // sqrt(dx*dx + dy*dy), no contraction (numpy has none)
  return FM_SQRT64(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
}

template <int N, int OT>
__device__ __forceinline__ void f_load(const FormParams& p, int b, FEnv<N>& e) {
  const int O = OT >= 0 ? OT : p.O;
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) {
    const size_t k = (size_t)b * N + i;
    e.px[i] = p.st.pos[2 * k]; e.py[i] = p.st.pos[2 * k + 1]; e.vx[i] = p.st.vel[2 * k]; e.vy[i] = p.st.vel[2 * k + 1];
    e.pd[i] = p.st.p_dist[k]; e.lx[i] = p.st.landmark_pos[2 * k]; e.ly[i] = p.st.landmark_pos[2 * k + 1];
    e.gm[i] = p.st.goal_match[k]; e.dtg[i] = p.st.dists_to_goal[k]; e.treq[i] = p.st.times_required[k];
    e.dleft[i] = p.st.dist_left_to_goal[k]; e.nac[i] = p.st.num_agent_collisions[k]; e.noc[i] = p.st.num_obstacle_collisions[k];
    e.mint[i] = p.st.min_time[k]; e.status[i] = p.st.status[k] != 0; e.reached[i] = p.st.goal_reached[k];
    e.occ[i] = p.st.occupied[k]; e.hist[i] = p.st.goal_history[k];
  }
  FM_UNROLL_O
  for (int k = 0; k < O; ++k) { e.ox[k] = p.st.obstacle_pos[((size_t)b * O + k) * 2]; e.oy[k] = p.st.obstacle_pos[((size_t)b * O + k) * 2 + 1]; }
  e.dmean = p.st.dist_traveled_mean[b]; e.dstd = p.st.dist_traveled_stddev[b]; e.step = p.st.step[b]; e.episode = p.st.episode[b];
  if constexpr (OT < 0) {                                                  // walls: generic instantiation only
    for (int w = 0; w < p.W; ++w) { e.wax[w] = p.st.wall_axis[(size_t)b * p.W + w]; e.wor[w] = p.st.wall_orient[(size_t)b * p.W + w]; }
    if (p.W) e.wlen = p.st.wall_len[b];
  }
}

template <int N, int OT>
__device__ __forceinline__ void f_store(const FormParams& p, int b, const FEnv<N>& e, bool statics) {
  const int O = OT >= 0 ? OT : p.O;
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) {
    const size_t k = (size_t)b * N + i;
    p.st.pos[2 * k] = (float)e.px[i]; p.st.pos[2 * k + 1] = (float)e.py[i]; p.st.vel[2 * k] = (float)e.vx[i]; p.st.vel[2 * k + 1] = (float)e.vy[i];
    p.st.p_dist[k] = (float)e.pd[i]; p.st.goal_match[k] = e.gm[i]; p.st.dists_to_goal[k] = (float)e.dtg[i];
    p.st.times_required[k] = (float)e.treq[i]; p.st.dist_left_to_goal[k] = (float)e.dleft[i];
    p.st.num_agent_collisions[k] = e.nac[i]; p.st.num_obstacle_collisions[k] = e.noc[i];
    p.st.min_time[k] = e.mint[i]; p.st.status[k] = e.status[i] ? 1 : 0; p.st.goal_reached[k] = e.reached[i];
    p.st.occupied[k] = (float)e.occ[i]; p.st.goal_history[k] = e.hist[i];
    if (statics) { p.st.landmark_pos[2 * k] = e.lx[i]; p.st.landmark_pos[2 * k + 1] = e.ly[i]; }
  }
  if (statics) {
    FM_UNROLL_O
    for (int k = 0; k < O; ++k) { p.st.obstacle_pos[((size_t)b * O + k) * 2] = e.ox[k]; p.st.obstacle_pos[((size_t)b * O + k) * 2 + 1] = e.oy[k]; }
    if constexpr (OT < 0) {
      for (int w = 0; w < p.W; ++w) { p.st.wall_axis[(size_t)b * p.W + w] = e.wax[w]; p.st.wall_orient[(size_t)b * p.W + w] = e.wor[w]; }
      if (p.W) p.st.wall_len[b] = e.wlen;
    }
  }
  p.st.dist_traveled_mean[b] = (float)e.dmean; p.st.dist_traveled_stddev[b] = (float)e.dstd; p.st.step[b] = e.step; p.st.episode[b] = e.episode;
}

template <int N>
__device__ __forceinline__ void f_dists(FEnv<N>& e) {
  FM_UNROLL_N
  for (int a = 0; a < N; ++a) {
    FM_UNROLL_N
    for (int g = 0; g < N; ++g) e.dal[a * N + g] = dn(e.px[a] - (double)e.lx[g], e.py[a] - (double)e.ly[g]);
  }
}

// is_obstacle_collision (:576-586, no walls): closer than 2.0 * (size + size) to any obstacle.
template <int N, int OT>
__device__ __forceinline__ bool f_obstacle_hit(const FormParams& p, const FEnv<N>& e, double x, double y) {
  const int O = OT >= 0 ? OT : p.O;
  const double dmin = 2.0 * (0.05 + 0.05);
  bool hit = false;
  FM_UNROLL_O
  for (int k = 0; k < O; ++k) hit = hit || (dn((double)e.ox[k] - x, (double)e.oy[k] - y) < dmin);
  if constexpr (OT < 0) {                                                  // :588-600: inside a wall's box grown by 1.5 * size
    for (int w = 0; w < p.W; ++w) {
      const double prll = e.wor[w] == 0 ? x : y, perp = e.wor[w] == 0 ? y : x, ax = (double)e.wax[w], wl = (double)e.wlen, g = 1.5 * 0.05;
      hit = hit || ((ax - g) <= perp && perp <= (ax + g) && (-wl - g) <= prll && prll <= (wl + g));
    }
  }
  return hit;
}

// np.mean / np.std (population) of a length-N vector.
template <int N>
__device__ __forceinline__ void f_mean_std(const double (&v)[N], double& mean, double& sd) {
  double s = 0.0;
  FM_UNROLL_N
  for (int j = 0; j < N; ++j) s = __dadd_rn(s, v[j]);
  mean = FM_DIV64(s, (double)N);
  double q = 0.0;
  FM_UNROLL_N
  for (int j = 0; j < N; ++j) { const double d = v[j] - mean; q = __dadd_rn(q, __dmul_rn(d, d)); }
  sd = FM_SQRT64(FM_DIV64(q, (double)N));
}

// Far branch shared by observation (:933-956) and the agent rows of the node features (:1256-1270): nearest goal not
// marked occupied (== 1); if every goal is, the entity itself and a cleared table.  (qx, qy) = position of agent a, `a` and
// `slot` compile-time values after unrolling.
template <int N>
__device__ __forceinline__ int f_pick_goal(FEnv<N>& e, int a, double qx, double qy, int slot, double& gx, double& gy, double& occ, float& hist) {
  int best = -1;
  double bd = 0.0, bx = 0.0, by = 0.0, bo = 0.0;
  float bh = 0.0f;
  FM_UNROLL_N
  for (int g = 0; g < N; ++g) {
    const double d = e.dal[a * N + g];
    const bool take = e.occ[g] != 1.0 && (best < 0 || d < bd);
    if (take) { best = g; bd = d; bx = (double)e.lx[g]; by = (double)e.ly[g]; bo = e.occ[g]; bh = e.hist[g]; }
  }
  if (best >= 0) { gx = bx; gy = by; occ = bo; hist = bh; return best; }
  FM_UNROLL_N
  for (int g = 0; g < N; ++g) e.occ[g] = 0.0;                              // :951 / :1266
  gx = qx; gy = qy; occ = e.occ[slot]; hist = e.hist[slot];
  return -1;
}

// Scenario.observation (:840-1015) of agent i: 11 values, updates the occupancy table and the goal history.
template <int N>
__device__ __forceinline__ void f_observation(const FormParams& p, FEnv<N>& e, int i, float* __restrict__ o) {
  const double x = e.px[i], y = e.py[i];
  double d[N];
  int first = 0;
  double mind = e.dal[i * N];
  FM_UNROLL_N
  for (int g = 0; g < N; ++g) { d[g] = e.dal[i * N + g]; if (d[g] < mind) { first = g; mind = d[g]; } }
  int second = first == 0 ? 1 : 0;                                         // np.argsort(dists)[1]
  double dsec = first == 0 ? d[N > 1 ? 1 : 0] : d[0];
  FM_UNROLL_N
  for (int g = 0; g < N; ++g) if (g != first && d[g] < dsec) { second = g; dsec = d[g]; }
  const double sgx = (double)ld(e.lx, second), sgy = (double)ld(e.ly, second), socc = ld(e.occ, second);   // read before the updates below
  const double th = p.min_dist_thresh;
  double gx, gy, gocc;
  float ghist;
  if (mind < p.min_obs_dist) {
    int chosen = first;
    gx = (double)ld(e.lx, chosen); gy = (double)ld(e.ly, chosen);
    FM_UNROLL_N
    for (int g = 0; g < N; ++g) {                                          // :866-879 nearby goals marked occupied
      if (!(d[g] < p.min_obs_dist) || e.occ[g] != 1.0) continue;
      bool any = false; double mn = 0.0;
      FM_UNROLL_N
      for (int j = 0; j < N; ++j) { const double q = e.dal[j * N + g]; any = any || (q < th); mn = j == 0 ? q : fmin(mn, q); }
      if (!any) e.occ[g] = mn;
    }
    if (mind < th) {                                                       // :882-885
      st(e.occ, chosen, 1.0); st(e.hist, chosen, (float)i);
    } else {
      bool any = false; double closest = 0.0;
      FM_UNROLL_N
      for (int j = 0; j < N; ++j) { const double q = ldm<N>(e.dal, j, chosen); any = any || (q < th); closest = j == 0 ? q : fmin(closest, q); }
      if (ld(e.occ, chosen) == 1.0 && any) {                               // :908-923: nearest FREE goal; `chosen` becomes its
        int k = 0, bestk = -1; double bd = 0.0, bx = 0.0, by = 0.0;        //   index in the free SUBSET (reference quirk, kept)
        FM_UNROLL_N
        for (int g = 0; g < N; ++g) {
          if (e.occ[g] == 1.0) continue;
          const double q = d[g];
          if (bestk < 0 || q < bd) { bestk = k; bd = q; bx = (double)e.lx[g]; by = (double)e.ly[g]; }
          ++k;
        }
        if (bestk >= 0) { chosen = bestk; gx = bx; gy = by; }              // (no free goal: the reference raises)
      } else {
        st(e.occ, chosen, 1.0 - closest);
      }
    }
    gocc = ld(e.occ, chosen); ghist = ld(e.hist, chosen);                  // :930-931
  } else {
    f_pick_goal<N>(e, i, x, y, i, gx, gy, gocc, ghist);
  }
  if (o) {
    o[0] = (float)e.vx[i]; o[1] = (float)e.vy[i]; o[2] = (float)x; o[3] = (float)y; o[4] = (float)(gx - x); o[5] = (float)(gy - y);
    o[6] = (float)gocc; o[7] = ghist; o[8] = (float)(sgx - x); o[9] = (float)(sgy - y); o[10] = (float)socc;
  }
}

// graph_observation + _get_entity_feat_relative (:1083-1178, :1222-1340) for ego agent i, as a RECIPE: per agent a the goal
// it is shown heading for with that goal's occupancy / history (the far branch may clear the occupancy table, :1266).  The
// velocities ego i sees are the post-integration ones with the agents that latched at ego index <= i zeroed (rec latch[]).
template <int N, int OT>
__device__ __forceinline__ void f_node_recipe(const FormParams& p, FEnv<N>& e, int i, float* __restrict__ rec) {
  const int O = OT >= 0 ? OT : p.O, W = OT >= 0 ? 0 : p.W;
  float* pk = rec + 2 * (2 * N + O + W) + 3 * N + i * 3 * N;
  FM_UNROLL_N
  for (int a = 0; a < N; ++a) {
    const double qx = e.px[a], qy = e.py[a];
    int first = 0; double mind = 0.0, focc = 0.0; float fhist = 0.0f;
    FM_UNROLL_N
    for (int g = 0; g < N; ++g) { const double d = e.dal[a * N + g]; if (g == 0 || d < mind) { first = g; mind = d; focc = e.occ[g]; fhist = e.hist[g]; } }
    double gx, gy, occ;
    float hist;
    int gi = first;
    if (mind < p.min_obs_dist) { occ = focc; hist = fhist; }
    else gi = f_pick_goal<N>(e, a, qx, qy, a, gx, gy, occ, hist);
    pk[3 * a] = (float)gi; pk[3 * a + 1] = (float)occ; pk[3 * a + 2] = hist;
  }
}

// head of the recipe: positions of the E entities (agents, landmarks, obstacles), velocities, no latch yet
template <int N, int OT>
__device__ __forceinline__ void f_rec_head(const FormParams& p, const FEnv<N>& e, float* __restrict__ rec) {
  const int O = OT >= 0 ? OT : p.O;
  FM_UNROLL_N
  for (int a = 0; a < N; ++a) {
    rec[2 * a] = (float)e.px[a]; rec[2 * a + 1] = (float)e.py[a];
    rec[2 * (N + a)] = e.lx[a]; rec[2 * (N + a) + 1] = e.ly[a];
  }
  FM_UNROLL_O
  for (int k = 0; k < O; ++k) { rec[2 * (2 * N + k)] = e.ox[k]; rec[2 * (2 * N + k) + 1] = e.oy[k]; }
  int W = 0;
  if constexpr (OT < 0) {
    W = p.W;
    for (int w = 0; w < W; ++w) {                                          // wall.state.p_pos (:316-333): the midpoint
      rec[2 * (2 * N + O + w)] = e.wor[w] == 0 ? 0.0f : e.wax[w]; rec[2 * (2 * N + O + w) + 1] = e.wor[w] == 0 ? e.wax[w] : 0.0f;
    }
    if (W) { float* x = rec + 2 * (2 * N + O + W) + 3 * N + 3 * N * N; x[0] = e.wlen; x[1] = e.wax[0]; x[2] = W > 1 ? e.wax[1] : 0.0f; }
  }
  float* v = rec + 2 * (2 * N + O + W);
  FM_UNROLL_N
  for (int a = 0; a < N; ++a) { v[2 * a] = (float)e.vx[a]; v[2 * a + 1] = (float)e.vy[a]; v[2 * N + a] = (float)(N + 1); }
}

// One node_obs row (ego agent i, entity en) from an env's recipe (:1222-1340):
//   [v_e - v_i (2), p_e - p_i (2), goal_e - p_i (2), goal occupied, goal history, p_e - p_i (2), p_e - p_i (2), type]
// landmarks: occupied 1, history = landmark id; obstacles: occupied 1, history 0 (id None); both with v_e = 0, goal = p_e.
// Walls (:1323-1334; W > 0, the last W entities): p_e = the midpoint, the two trailing pairs are the corner offsets
// (-len, axis + width / 2) - p_i and (len, axis - width / 2) - p_i as (x, y) whatever the orientation, type 3, history =
// wall id in the fair-assignment files (wall_hist 1) and 0 in the base scenarios.
__device__ __forceinline__ void f_row(const float* __restrict__ rec, int N, int O, int i, int en, float* __restrict__ q,
                                      int W = 0, int wall_hist = 0) {
  const float* v = rec + 2 * (2 * N + O + W);
  const float* latch = v + 2 * N;
  const float* pk = latch + N + i * 3 * N;
  const bool zi = latch[i] <= (float)i;
  const float x = rec[2 * i], y = rec[2 * i + 1], vx = zi ? 0.0f : v[2 * i], vy = zi ? 0.0f : v[2 * i + 1];
  const float rx = rec[2 * en] - x, ry = rec[2 * en + 1] - y;
  float rvx = 0.0f - vx, rvy = 0.0f - vy, gx = rx, gy = ry, occ = 1.0f, hist = 0.0f, type = 2.0f;
  float c0 = rx, c1 = ry, c2 = rx, c3 = ry;
  if (en < N) {
    const bool ze = latch[en] <= (float)i;
    rvx = (ze ? 0.0f : v[2 * en]) - vx; rvy = (ze ? 0.0f : v[2 * en + 1]) - vy;
    const int gi = (int)pk[3 * en];
    if (gi >= 0) { gx = rec[2 * (N + gi)] - x; gy = rec[2 * (N + gi) + 1] - y; }      // gi < 0: the agent's own position (rel pos)
    occ = pk[3 * en + 1]; hist = pk[3 * en + 2]; type = 0.0f;
  } else if (en < 2 * N) {
    hist = (float)(en - N); type = 1.0f;
  } else if (en >= 2 * N + O) {
    const int w = en - (2 * N + O);
    const float* wx = pk - i * 3 * N + 3 * N * N;                          // (half-length, axis 0, axis 1)
    c0 = -wx[0] - x; c1 = (wx[1 + w] + 0.05f) - y; c2 = wx[0] - x; c3 = (wx[1 + w] - 0.05f) - y;
    hist = wall_hist ? (float)w : 0.0f; type = 3.0f;
  }
  q[0] = rvx; q[1] = rvy; q[2] = rx; q[3] = ry; q[4] = gx; q[5] = gy; q[6] = occ; q[7] = hist;
  q[8] = c0; q[9] = c1; q[10] = c2; q[11] = c3; q[12] = type;
}

// One entry of cached_dist_mag (core.py:204-228) = adj [E, E], from the recipe's fp32 positions (the positions the state
// block stores), float64 distance rounded once.
__device__ __forceinline__ float f_adj_elem(const float* __restrict__ rec, int a, int c) {
  return a == c ? 0.0f : (float)dn((double)rec[2 * a] - (double)rec[2 * c], (double)rec[2 * a + 1] - (double)rec[2 * c + 1]);
}

// Lexifair by sorted threshold descent for one thread (marl_fair_assign.py:16-55; oracle/lexifair.py lexifair_descent; the
// group-parallel form is lexifair_group<G>, fm_device.cuh): entries are visited from the largest key (cost, i, j) down; an
// entry is deleted unless the remaining entries would lose their perfect matching, in which case it is the bottleneck of
// every remaining solution and its row / column freeze.  N <= 8: row masks are bytes, augmenting paths by depth-first search.
template <int N>
__device__ void lexifair_serial(const double (&c)[N * N], int (&out)[N]) {
  unsigned char ord[N * N];
  for (int k = 0; k < N * N; ++k) {                                        // insertion sort, descending by (cost, flat index)
    int q = k;
    while (q > 0 && (c[ord[q - 1]] < c[k] || (c[ord[q - 1]] == c[k] && ord[q - 1] < k))) { ord[q] = ord[q - 1]; --q; }
    ord[q] = (unsigned char)k;
  }
  unsigned rowmask[N];
  int match[N], colrow[N];
  bool frozen[N];
  for (int r = 0; r < N; ++r) { rowmask[r] = (1u << N) - 1u; match[r] = r; colrow[r] = r; frozen[r] = false; }
  for (int t = 0; t < N * N; ++t) {
    const int r = ord[t] / N, col = ord[t] % N;
    if (!((rowmask[r] >> col) & 1u)) continue;
    rowmask[r] &= ~(1u << col);
    if (match[r] != col) continue;                                         // the matching survives the deletion
    // row r and column col are free: look for an augmenting path r -> ... -> col (iterative DFS over rows)
    int stack_row[N], stack_it[N], via[N];                                 // via[c]: row that reached column c
    unsigned seen = 0;
    int sp = 0;
    stack_row[0] = r; stack_it[0] = 0;
    bool found = false;
    while (sp >= 0 && !found) {
      const int rr = stack_row[sp];
      int cc = stack_it[sp];
      while (cc < N && (!((rowmask[rr] >> cc) & 1u) || ((seen >> cc) & 1u))) ++cc;
      if (cc >= N) { --sp; continue; }
      stack_it[sp] = cc + 1;
      seen |= 1u << cc;
      via[cc] = rr;
      if (cc == col) { found = true; break; }
      const int owner = colrow[cc];
      if (frozen[owner]) continue;                                         // (a frozen row's column was removed from every mask)
      ++sp; stack_row[sp] = owner; stack_it[sp] = 0;
    }
    if (found) {                                                           // flip the path back from `col`
      int cc = col;
      while (true) {
        const int rr = via[cc];
        const int prev = match[rr];                                        // column rr gives up (== -1 for the start row r)
        match[rr] = cc; colrow[cc] = rr;
        if (rr == r) break;
        cc = prev;
      }
    } else {                                                               // critical entry: freeze row r / column col
      rowmask[r] = 0u; frozen[r] = true; match[r] = col; colrow[col] = r;
      for (int q = 0; q < N; ++q) if (q != r) rowmask[q] &= ~(1u << col);
    }
  }
  for (int r = 0; r < N; ++r) out[r] = match[r];
}

// cdist(agent_pos, goal_pos) + lexifair (:704-721, :481-486); the costs are the step's distance matrix
template <int N>
__device__ __forceinline__ void f_assign(FEnv<N>& e) {
  if constexpr (N <= 4) {
    lexifair_small<N>(e.dal, e.gm);
  } else {
    double c[N * N];
    for (int k = 0; k < N * N; ++k) c[k] = e.dal[k];
    lexifair_serial<N>(c, e.gm);
  }
}

// Min-sum matching of the current agent -> goal distances by enumeration (scipy linear_sum_assignment in
// nav_base_formation_graph_mask.py:255-260 and :686-689): match[i] = goal of agent i, delta[i] its distance.  N <= 5
// (larger teams: f_min_sum_sap below).
// Takes a COPY of the cost matrix (not the env: the env must not escape to a function that is not inlined).
template <int N>
__device__ __noinline__ void f_min_sum_c(const double* __restrict__ cin, int* __restrict__ match, double* __restrict__ delta) {
  double c[N * N];
  for (int k = 0; k < N * N; ++k) c[k] = cin[k];
  int perm[N], best[N];
  for (int i = 0; i < N; ++i) { perm[i] = i; best[i] = i; }
  double bs = 0.0;
  bool have = false;
  while (true) {                                                           // permutations in lexicographic order
    double sum = 0.0;
    for (int i = 0; i < N; ++i) sum += c[i * N + perm[i]];
    if (!have || sum < bs) { bs = sum; have = true; for (int i = 0; i < N; ++i) best[i] = perm[i]; }
    int k = N - 2;
    while (k >= 0 && perm[k] > perm[k + 1]) --k;
    if (k < 0) break;
    int l = N - 1;
    while (perm[l] < perm[k]) --l;
    int t = perm[k]; perm[k] = perm[l]; perm[l] = t;
    for (int a = k + 1, b = N - 1; a < b; ++a, --b) { t = perm[a]; perm[a] = perm[b]; perm[b] = t; }
  }
  for (int i = 0; i < N; ++i) { match[i] = best[i]; delta[i] = c[i * N + best[i]]; }
}
// Min-sum matching for N >= 6, where N! permutations per step are too many: scipy's shortest augmenting path
// (rectangular_lsap.cpp after Crouse 2016, square case; oracle/lsap.py states it) with its operation order and tie rule,
// so that match equals scipy's col_ind bit for bit, ties included.  One thread, local arrays; a COPY of the cost matrix
// like f_min_sum_c.  The warp-per-problem form of the same loop is lsap_kernel (fm_lsap.cu).
template <int N>
__device__ __noinline__ void f_min_sum_sap(const double* __restrict__ cin, int* __restrict__ match, double* __restrict__ delta) {
  double c[N * N], u[N], v[N], spc[N];
  int col4row[N], row4col[N], path[N], rem[N];
  bool sr[N], sc[N];
  for (int k = 0; k < N * N; ++k) c[k] = cin[k];
  for (int k = 0; k < N; ++k) { u[k] = 0.0; v[k] = 0.0; col4row[k] = -1; row4col[k] = -1; path[k] = -1; }
  for (int cur = 0; cur < N; ++cur) {
    for (int k = 0; k < N; ++k) { rem[k] = N - 1 - k; sr[k] = false; sc[k] = false; spc[k] = INFINITY; }
    double minv = 0.0;
    int nrem = N, i = cur, sink = -1;
    while (sink == -1) {
      sr[i] = true;
      int index = 0;                     // always set below: an unassigned column stays in rem, and spc is never NaN
      double lowest = INFINITY;
      for (int it = 0; it < nrem; ++it) {
        const int j = rem[it];
        const double r = minv + c[i * N + j] - u[i] - v[j];       // adds only (nothing to contract), scipy's order
        if (r < spc[j]) { path[j] = i; spc[j] = r; }
        if (spc[j] < lowest || (spc[j] == lowest && row4col[j] == -1)) { lowest = spc[j]; index = it; }
      }
      minv = lowest;
      const int j = rem[index];
      if (row4col[j] == -1) sink = j; else i = row4col[j];
      sc[j] = true;
      rem[index] = rem[--nrem];
    }
    u[cur] += minv;
    for (int r = 0; r < N; ++r)
      if (sr[r] && r != cur) u[r] += minv - spc[col4row[r]];
    for (int j = 0; j < N; ++j)
      if (sc[j]) v[j] -= minv - spc[j];
    for (int j = sink;;) {                                                 // augment along path[] back to row cur
      const int r = path[j];
      row4col[j] = r;
      const int t = col4row[r]; col4row[r] = j; j = t;
      if (r == cur) break;
    }
  }
  for (int r = 0; r < N; ++r) { match[r] = col4row[r]; delta[r] = c[r * N + col4row[r]]; }
}
template <int N>
__device__ __forceinline__ void f_min_sum(const FEnv<N>& e, int (&match)[N], double (&delta)[N]) {
  double c[N * N], dl[N];
  int m[N];
  FM_UNROLL_N
  for (int k = 0; k < N * N; ++k) c[k] = e.dal[k];
  if constexpr (N >= 6) f_min_sum_sap<N>(c, m, dl);
  else f_min_sum_c<N>(c, m, dl);
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) { match[i] = m[i]; delta[i] = dl[i]; }
}

// env.reset()'s observation pass (environment.py:882-898): obs_i, then node rows_i, per agent.
template <int N, int OT>
__device__ __forceinline__ void f_observe(const FormParams& p, FEnv<N>& e, const FOut& o) {
  f_rec_head<N, OT>(p, e, o.rec);
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) {
    f_observation<N>(p, e, i, o.obs + i * F_OBS);
    f_node_recipe<N, OT>(p, e, i, o.rec);
  }
}

// what a reset leaves in the per-agent latches, counters and tables (:217-288)
template <int N>
__device__ __forceinline__ void f_reset_init(FEnv<N>& e) {
  for (int i = 0; i < N; ++i) {
    e.vx[i] = e.vy[i] = 0.0; e.pd[i] = 0.0; e.status[i] = false; e.treq[i] = e.dtg[i] = e.dleft[i] = -1.0;
    e.noc[i] = e.nac[i] = 0.0f; e.hist[i] = -1.0f; e.reached[i] = -1.0f; e.occ[i] = 0.0;
  }
  e.step = 0;
}

// reset_world + random_scenario (:217-487) with the Philox draw scheme of the navigation kernels: draw counter per
// (seed, global env, episode); obstacles 0.8 * U, agents U rejected vs obstacles (2.0x) / placed agents (1.05x), goals
// 0.8 * U rejected vs obstacles (2.0x) / placed goals (1.2x; 1.5x in the base scenarios).  Positions are float32 values,
// predicates float64.
template <int N>
__device__ void f_reset(const FormParams& p, int b, FEnv<N>& e) {
  const long long genv = p.env_offset + b;
  const float ws = (float)p.world_size, half = (float)(p.world_size / 2);
  uint32_t d = 0;
  auto draw = [&](float& x, float& y) {
    uint32_t c0 = d, c1 = (uint32_t)e.episode, c2 = (uint32_t)((unsigned long long)genv & 0xffffffffull),
             c3 = (uint32_t)((unsigned long long)genv >> 32);
    philox4x32_10(c0, c1, c2, c3, p.seed_lo, p.seed_hi);
    x = __fsub_rn(__fmul_rn(ws, u01_24(c0)), half); y = __fsub_rn(__fmul_rn(ws, u01_24(c1)), half);
    ++d;
  };
  for (int k = 0; k < p.O; ++k) { float x, y; draw(x, y); e.ox[k] = __fmul_rn(0.8f, x); e.oy[k] = __fmul_rn(0.8f, y); }
  if (p.W) {
    // :233-234 wall_length = U(0.2, 0.8) * ws / 4 per reset; :301-304 axis = +-U(0.2, 0.9) * ws / 2 (wall 0 at +, wall 1 at -);
    // :306 orientation per wall.  One draw each, the raw 24-bit uniform of its x component.
    auto uni = [&]() { float x, y; draw(x, y); return __fdiv_rn(__fadd_rn(x, half), ws); };
    e.wlen = __fmul_rn(__fadd_rn(0.2f, __fmul_rn(0.6f, uni())), (float)(p.world_size / 4));
    const float wp = __fmul_rn(__fadd_rn(0.2f, __fmul_rn(0.7f, uni())), half);
    for (int w = 0; w < p.W; ++w) { e.wax[w] = w == 0 ? wp : -wp; e.wor[w] = uni() >= 0.5f ? 1 : 0; }
  }
  const double r2 = 0.05 + 0.05;
  for (int pass = 0; pass < 2; ++pass) {
    double X[N], Y[N];
    const double dsame = pass ? (p.assignment == 0 ? 1.2 : 1.5) * r2 : 1.05 * r2;   // goals: :638-648; 1.5x in the base files
    for (int a = 0; a < N; ++a) {
      while (true) {
        float fx, fy; draw(fx, fy);
        if (pass) { fx = __fmul_rn(0.8f, fx); fy = __fmul_rn(0.8f, fy); }
        const double x = fx, y = fy;
        bool bad = f_obstacle_hit<N, -1>(p, e, x, y);
        for (int j = 0; j < a; ++j) bad = bad || (dn(X[j] - x, Y[j] - y) < dsame);
        if (!bad || d >= (uint32_t)MAX_DRAWS) {
          X[a] = x; Y[a] = y;
          if (pass) { e.lx[a] = fx; e.ly[a] = fy; } else { e.px[a] = x; e.py[a] = y; }
          break;
        }
      }
    }
  }
  f_dists<N>(e);
  f_reset_init<N>(e);
  for (int i = 0; i < N; ++i)
    if (p.has_max_speed) e.mint[i] = (float)(e.dal[i * N + i] / p.max_speed);   // goal_match = arange here (:229, :474-476)
  if (p.assignment == 0) {
    f_assign<N>(e);
  } else if (p.assignment == 1) {                                          // nav_base_formation_graph_mask.py:255-260
    double delta[N];
    f_min_sum<N>(e, e.gm, delta);
  } else {                                                                 // np.random.shuffle(arange) (randomgoal :258-259):
    for (int i = 0; i < N; ++i) e.gm[i] = i;                               // Fisher-Yates on the same draw stream
    for (int k = N - 1; k > 0; --k) {
      float x, y; draw(x, y);
      const float u = __fdiv_rn(__fadd_rn(x, half), ws);
      int j = (int)__fmul_rn(u, (float)(k + 1));
      j = j < k ? j : k;
      const int t = e.gm[k]; e.gm[k] = e.gm[j]; e.gm[j] = t;
    }
  }
  e.episode += 1;
}

// One softplus contact term (core.py:389-392, cached branch: dist_min = size + size): fp32 with hardware rsqrt / ex2 and
// the polynomial log1p of the navigation kernels (fm_device.cuh contact_force: relative error of the term ~5e-7).
__device__ __forceinline__ void f_pair_force(float dx, float dy, float& fx, float& fy, float dmin = 0.1f) {
  const float d2 = fmaf(dx, dx, __fmul_rn(dy, dy));
  const float inv = rsqrt_approx(d2);
  const float dist = __fmul_rn(d2, inv);
  const float x = __fmul_rn(__fsub_rn(dmin, dist), 50.0f);                 // -(dist - dist_min) / k,  k = 0.02
  const float t = ex2_approx(__fmul_rn(-fabsf(x), 1.4426950408889634f));
  const float sp = __fadd_rn(fmaxf(x, 0.0f), log1p_unit(t));
  const float c = __fmul_rn(__fmul_rn(6.0f, sp), inv);                     // contact_force (300) * k * softplus / dist
  fx = __fmul_rn(c, dx); fy = __fmul_rn(c, dy);
}

// get_wall_collision_force (core.py:407-462) of an agent at (px, py): wall_contact_force 220, margin 0.024, entity size
// 0.05, width 0.1; wall along x at y = axis ('H') or along y at x = axis, endpoints [-len, len].  float64 like the reference,
// so that the end-cap branches (where the force is discontinuous) are taken on the same side.
__device__ __forceinline__ void f_wall_force(double px, double py, bool horiz, float axis, float len, float& fx, float& fy) {
  const double prll = horiz ? px : py, perp = horiz ? py : px;
  const double l = (double)len, r = 0.05;
  if (prll < -l - r || prll > l + r) return;                               // beyond the endpoints: None (:417-419)
  double st = 0.0, ct = 1.0;                                               // sin / cos of theta
  if (prll < -l || prll > l) {                                             // part of the entity is past an end (:420-428)
    const double past = prll < -l ? prll + l : prll - l;
    st = past / r;                                                         // theta = arcsin(past / size)
    ct = sqrt(fmax(0.0, 1.0 - st * st));
  }
  const double dist_min = ct * r + 0.05;                                   // + 0.5 * width
  const double delta = perp - (double)axis;                                // :435
  const double dist = fabs(delta);
  const double k = 0.024;
  const double x = -(dist - dist_min) / k;
  const double pen = (fmax(x, 0.0) + log1p(exp(-fabs(x)))) * k;            // logaddexp(0, x) * k (:439)
  const double mag = 220.0 * delta / dist * pen;                           // :440
  const double fperp = ct * mag, fprll = st * fabs(mag);                   // :444-445
  fx += (float)(horiz ? fprll : fperp);
  fy += (float)(horiz ? fperp : fprll);
}

// ---- pending resets (split step path) -----------------------------------------------------------------------------------
// What a reset draws depends on (seed, global env, episode) only, so it can be computed AHEAD: formation_prefetch_kernel
// (fm_form_image.cu) runs f_reset for every env whose pending block is stale, beside the image kernel, and leaves
//   tag (the episode key the block was drawn for) | px py [N] | lx ly [N] | ox oy [O] | min_time [N] | goal_match [N]
// in a handle-owned SoA block ([field][Bp], lane = env: coalesced).  The auto-reset inside the step then only copies the
// block, clears the latches and re-observes.  Without this the step kernel's duration was set by the handful of warps in
// which some env finished early: one lane walking the serial rejection sampling (about 12 000 instructions from local
// memory) while 2 047 warps had long finished -- 53 us instead of 29 for the same instruction total (profiles/r02_n).
__host__ __device__ inline int form_pending_floats(int N, int O) { return 1 + 6 * N + 2 * O; }

#ifdef __CUDACC__
template <int N>
__device__ void f_pending_write(const FormParams& p, int b, const FEnv<N>& e, int key) {
  float* q = p.pend + b;
  const size_t S = (size_t)p.Bp;
  int f = 1;
  for (int i = 0; i < N; ++i) { q[f++ * S] = (float)e.px[i]; q[f++ * S] = (float)e.py[i]; }
  for (int i = 0; i < N; ++i) { q[f++ * S] = e.lx[i]; q[f++ * S] = e.ly[i]; }
  for (int k = 0; k < p.O; ++k) { q[f++ * S] = e.ox[k]; q[f++ * S] = e.oy[k]; }
  for (int i = 0; i < N; ++i) q[f++ * S] = e.mint[i];
  for (int i = 0; i < N; ++i) q[f++ * S] = __int_as_float(e.gm[i]);
  __threadfence();                                                         // a concurrent step kernel that sees the tag sees the block
  q[0] = __int_as_float(key);
}

// The reset of env b for episode key e.episode from its pending block; false (nothing touched) if the block is stale.
template <int N, int OT>
__device__ __forceinline__ bool f_pending_apply(const FormParams& p, int b, FEnv<N>& e) {
  const int O = OT >= 0 ? OT : p.O;
  const float* q = p.pend + b;
  const size_t S = (size_t)p.Bp;
  if (__float_as_int(q[0]) != e.episode) return false;
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) { e.px[i] = (double)q[(1 + 2 * i) * S]; e.py[i] = (double)q[(2 + 2 * i) * S]; }
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) { e.lx[i] = q[(1 + 2 * N + 2 * i) * S]; e.ly[i] = q[(2 + 2 * N + 2 * i) * S]; }
  FM_UNROLL_O
  for (int k = 0; k < O; ++k) { e.ox[k] = q[(1 + 4 * N + 2 * k) * S]; e.oy[k] = q[(2 + 4 * N + 2 * k) * S]; }
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) { const float m = q[(1 + 4 * N + 2 * O + i) * S]; if (p.has_max_speed) e.mint[i] = m; }
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) e.gm[i] = __float_as_int(q[(1 + 5 * N + 2 * O + i) * S]);
  f_dists<N>(e);
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) {
    e.vx[i] = e.vy[i] = 0.0; e.pd[i] = 0.0; e.status[i] = false; e.treq[i] = e.dtg[i] = e.dleft[i] = -1.0;
    e.noc[i] = e.nac[i] = 0.0f; e.hist[i] = -1.0f; e.reached[i] = -1.0f; e.occ[i] = 0.0;
  }
  e.step = 0;
  e.episode += 1;
  return true;
}
#endif  // __CUDACC__

// reset() path for one env: optional reset, observation pass.  Runs on the generic (runtime O) code: resets are rare.
template <int N>
__device__ void form_reset_env(const FormParams& p, int b, const FOut& o) {
  FEnv<N> e;
  f_load<N, -1>(p, b, e);
  const bool doit = !p.mask || p.mask[b] != 0;
  if (doit) f_reset<N>(p, b, e); else f_dists<N>(e);
  f_observe<N, -1>(p, e, o);
  f_store<N, -1>(p, b, e, doit);
}

// Auto-reset at the end of a step (env_wrappers.py:859-865), out of line with an env of its own: the step's env stays in
// registers (a reference handed to a call would give it a home in local memory for the whole step).  dist_traveled_mean /
// stddev are world attributes the reset does not touch.  Two forms: the generic one draws the reset here (serial rejection
// sampling, env in local memory); the fast one (split step path, pending block valid) copies the block and re-observes on the
// unrolled register code -- this is the path whose latency sets the logic kernel's duration whenever some env finishes early.
template <int N>
__device__ __noinline__ void form_reset_tail(const FormParams& p, int b, int episode, double dmean, double dstd, const FOut& o) {
  FEnv<N> e;
  e.episode = episode; e.dmean = dmean; e.dstd = dstd;
  for (int i = 0; i < N; ++i) e.mint[i] = p.st.min_time[(size_t)b * N + i];   // kept when max_speed is None
  f_reset<N>(p, b, e);
  f_observe<N, -1>(p, e, o);
  f_store<N, -1>(p, b, e, true);
}
#ifdef __CUDACC__
template <int N, int OT>
__device__ __noinline__ void form_reset_tail_fast(const FormParams& p, int b, int episode, double dmean, double dstd, const FOut& o) {
  FEnv<N> e;
  e.episode = episode; e.dmean = dmean; e.dstd = dstd;
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) e.mint[i] = p.st.min_time[(size_t)b * N + i];
  f_pending_apply<N, OT>(p, b, e);                                          // the caller checked the tag
  f_observe<N, OT>(p, e, o);
  f_store<N, OT>(p, b, e, true);
}
#endif

// MultiAgentGraphEnv.step (environment.py:816-877) + graphworker auto-reset (env_wrappers.py:856-865) for one env.
template <int N, int OT = -1>
__device__ __forceinline__ void form_step_env(const FormParams& p, int b, const FOut& o) {
  FEnv<N> e;
  f_load<N, OT>(p, b, e);
  const int O = OT >= 0 ? OT : p.O;
  e.step += 1;                                                             // :819, :823
  // ---- World.step: action force (core.py:277-298), pair forces from the positions at step entry (:301-316, :370-404),
  // summed per agent in ascending partner order, joined to the float64 action force
  float cfx[N], cfy[N];
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) { cfx[i] = 0.f; cfy[i] = 0.f; }
  FM_UNROLL_N
  for (int a = 0; a < N; ++a) {
    FM_UNROLL_N
    for (int c = a + 1; c < N; ++c) {
      float fx, fy; f_pair_force((float)e.px[a] - (float)e.px[c], (float)e.py[a] - (float)e.py[c], fx, fy);
      if (!e.status[a]) { cfx[a] += fx; cfy[a] += fy; }                    // core.py:397
      if (!e.status[c]) { cfx[c] -= fx; cfy[c] -= fy; }                    // core.py:398
    }
    FM_UNROLL_O
    for (int k = 0; k < O; ++k) {                                          // obstacles: whatever the status (:401)
      float fx, fy; f_pair_force((float)e.px[a] - e.ox[k], (float)e.py[a] - e.oy[k], fx, fy);
      cfx[a] += fx; cfy[a] += fy;
    }
    if constexpr (OT < 0) {
      for (int w = 0; w < p.W; ++w) {                                      // a wall is also a circle entity of size = its width
        const float mx = e.wor[w] == 0 ? 0.0f : e.wax[w], my = e.wor[w] == 0 ? e.wax[w] : 0.0f;   // at its midpoint (core.py:186, :215)
        float fx, fy; f_pair_force((float)e.px[a] - mx, (float)e.py[a] - my, fx, fy, 0.05f + 0.1f);
        cfx[a] += fx; cfy[a] += fy;
      }
      for (int w = 0; w < p.W; ++w) f_wall_force(e.px[a], e.py[a], e.wor[w] == 0, e.wax[w], e.wlen, cfx[a], cfy[a]);   // core.py:317-327
    }
  }
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) {                                            // integrate_state (:338-356): every agent
    const int a = p.actions[(size_t)b * N + i];
    const double ux = (((a == 1) ? 1.0 : 0.0) - ((a == 2) ? 1.0 : 0.0)) * 5.0;   // environment.py:301-311
    const double uy = (((a == 3) ? 1.0 : 0.0) - ((a == 4) ? 1.0 : 0.0)) * 5.0;
    const double Fx = __dadd_rn(ux, (double)cfx[i]), Fy = __dadd_rn(uy, (double)cfy[i]);
    double vx = __dmul_rn(e.vx[i], 0.75), vy = __dmul_rn(e.vy[i], 0.75);
    vx = __dadd_rn(vx, __dmul_rn(Fx, 0.1)); vy = __dadd_rn(vy, __dmul_rn(Fy, 0.1));
    if (p.has_max_speed) {
      const double sp = dn(vx, vy);
      if (sp > p.max_speed) { vx = __dmul_rn(FM_DIV64(vx, sp), p.max_speed); vy = __dmul_rn(FM_DIV64(vy, sp), p.max_speed); }
    }
    e.vx[i] = vx; e.vy[i] = vy;
    const double sx = __dmul_rn(vx, 0.1), sy = __dmul_rn(vy, 0.1);
    e.px[i] = __dadd_rn(e.px[i], sx); e.py[i] = __dadd_rn(e.py[i], sy);
    e.pd[i] = __dadd_rn(e.pd[i], dn(sx, sy));
  }
  f_dists<N>(e);
  f_rec_head<N, OT>(p, e, o.rec);
  float* latch = o.rec + 2 * (2 * N + O + (OT >= 0 ? 0 : p.W)) + 2 * N;
  // info rows are written after the loop (only then is "every agent done" known): what a row holds is the agent's own
  // final state except the team statistics as they stood after ITS info_callback, kept here (6 floats per agent)
  float istat[N][6];
  const bool want_info = p.out.info != nullptr;

  // ---- per-agent loop (environment.py:832-864): observation, reward, node rows, done, info -- in this order
  double rew[N], delta[N];
  bool done[N], all_done = true;
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) delta[i] = 0.0;
  const double th = p.min_dist_thresh, dcoll = 1.05 * (0.05 + 0.05);
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) {
    f_observation<N>(p, e, i, o.obs + i * F_OBS);
    // reward (:691-802)
    double fairness;
    if (e.dtg[i] == -1.0) { double m, s; f_mean_std<N>(e.pd, m, s); fairness = FM_DIV64(m, s + 0.0001); }
    else fairness = FM_DIV64(e.dmean, e.dstd + 0.0001);
    if (i == 0 && p.assignment == 0) f_assign<N>(e);                       // :704-721: re-assignment every step
    if (i == 0 && p.assignment == 1) { int m[N]; f_min_sum<N>(e, m, delta); }   // mask.py:666-706 (the stored match stays)
    const double x = e.px[i], y = e.py[i];
    const double dg = p.assignment == 1 ? delta[i] : ldm<N>(e.dal, i, e.gm[i]);
    double r = 0.0;
    if (dg < th) {                                                         // :725-733
      if (!e.status[i]) { e.status[i] = true; e.vx[i] = 0.0; e.vy[i] = 0.0; latch[i] = (float)i; r += p.goal_rew; }
    } else {
      r -= dg;
    }
    int hits = 0;
    FM_UNROLL_N
    for (int j = 0; j < N; ++j) if (j != i && dn(e.px[j] - x, e.py[j] - y) < dcoll) { r -= p.collision_rew; ++hits; }
    const bool ohit = f_obstacle_hit<N, OT>(p, e, x, y);
    if (ohit) r -= p.collision_rew;
    if (p.fairness_reward) {                                               // :770-786
      double fair = p.fair_rew * tanh(fairness - p.zeroshift);
      if (fair < -p.fair_rew) fair = -p.fair_rew;
      r += fair;
    }
    r = fmin(fmax(r, -2.0 * p.collision_rew), p.goal_rew + p.fair_rew);
    rew[i] = r;
    f_node_recipe<N, OT>(p, e, i, o.rec);
    done[i] = e.status[i] || e.step >= p.episode_length;                   // environment.py:237-247
    all_done = all_done && done[i];
    // info_callback (:489-575)
    {
      int near = 0; double d = 0.0;
      FM_UNROLL_N
      for (int g = 0; g < N; ++g) { const double q = e.dal[i * N + g]; if (g == 0 || q < d) { near = g; d = q; } }
      const double now = (double)e.step * 0.1;
      const float nr = (float)near;
      if (d < th && (nr != e.reached[i] && e.reached[i] != -1.0f)) { e.reached[i] = nr; e.dleft[i] = d; }         // :497-499
      if (d < th && e.treq[i] == -1.0) { e.treq[i] = now; e.dtg[i] = e.pd[i]; e.dleft[i] = d; e.reached[i] = nr; }   // :501-505
      if (e.treq[i] == -1.0) { e.dtg[i] = e.pd[i]; e.dleft[i] = d; }                                                // :507-509
      if (d > th && e.treq[i] != -1.0) { e.dtg[i] = e.pd[i]; e.treq[i] = now; e.dleft[i] = d; }                      // :511-514
      if (d < th && nr == e.reached[i]) { e.dleft[i] = d; e.reached[i] = nr; }                                      // :516-518
      if (ohit) e.noc[i] += 1.0f;                                                                                   // :521-523
      e.nac[i] += (float)hits;
      f_mean_std<N>(e.dtg, e.dmean, e.dstd);                                                                        // :534-535
      if (want_info) {
        double tm, ts; f_mean_std<N>(e.treq, tm, ts);
        istat[i][0] = (float)e.dmean; istat[i][1] = (float)e.dstd; istat[i][2] = (float)FM_DIV64(e.dmean, e.dstd + 0.0001);
        istat[i][3] = (float)tm; istat[i][4] = (float)ts; istat[i][5] = (float)FM_DIV64(tm, ts + 0.0001);
      }
    }
  }
  double total = 0.0;
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) total += rew[i];
  FM_UNROLL_N
  for (int i = 0; i < N; ++i) {
    o.rew[i] = (float)(p.collaborative ? total : rew[i]);                  // environment.py:867-870
    o.done[i] = done[i] ? 1 : 0;
  }
  // info rows go straight to global memory, on the steps whose values the runner reads (every agent done; or every step)
  if (want_info && (all_done || p.info_every_step)) {
    FM_UNROLL_N
    for (int i = 0; i < N; ++i) {
      float* q = p.out.info + ((size_t)b * N + i) * INFO_F;
      q[0] = (float)rew[i]; q[1] = (float)e.dleft[i]; q[2] = (float)e.treq[i]; q[3] = e.nac[i]; q[4] = e.noc[i];
      q[5] = istat[i][0]; q[6] = istat[i][1]; q[7] = istat[i][2]; q[8] = (float)e.dtg[i];
      q[9] = (float)e.treq[i]; q[10] = istat[i][3]; q[11] = istat[i][4]; q[12] = istat[i][5]; q[13] = e.mint[i];
    }
  }
  if (p.auto_reset && all_done) {                                          // env_wrappers.py:859-865
#ifdef __CUDACC__
    if (OT >= 0 && p.pend && __float_as_int(p.pend[b]) == e.episode) form_reset_tail_fast<N, OT>(p, b, e.episode, e.dmean, e.dstd, o);
    else
#endif
      form_reset_tail<N>(p, b, e.episode, e.dmean, e.dstd, o);
  } else {
    f_store<N, OT>(p, b, e, false);
  }
}

// ---- device only from here: the shared-memory tile of a warp (tests/test_kernel_source_host.py cuts the host unit above this line)
#ifdef __CUDACC__
struct FormTile {            // floats per warp; all offsets multiples of 4 floats
  int obs, rew, done, rec, stage, rec_stride, words;
};
// with_stage: the fused kernel's two staging buffers (the logic kernel of the split path emits no rows: 3.3 KB less)
__host__ __device__ inline FormTile form_tile(int N, int O, int W = 0, bool with_stage = true) {
  FormTile t;
  t.stage = 0;                                                             // two staging buffers of F_CHUNK_WORDS
  t.obs = with_stage ? 2 * F_CHUNK_WORDS : 0;
  t.rew = t.obs + ((32 * N * F_OBS + 3) & ~3);
  t.done = t.rew + ((32 * N + 3) & ~3);
  t.rec = t.done + ((8 * N + 3) & ~3);                                      // 32 N bytes
  t.rec_stride = form_rec_floats(N, O, W) | 1;                                 // odd: lane = env accesses are conflict free
  t.words = t.rec + ((32 * t.rec_stride + 3) & ~3);
  return t;
}

#endif  // __CUDACC__

}  // namespace fm
