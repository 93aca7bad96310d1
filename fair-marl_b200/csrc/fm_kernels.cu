// Kernels of the B200-native navigation_graph simulator (compiled for sm_100a only).
//
//   step_kernel<G>    fused env step: action decode -> forces -> integration -> E x E distances ->
//                     per-agent observation / reward / info latches in the reference's sequential
//                     order -> done -> auto-reset (randomised placement + lexifair assignment) ->
//                     node features, adjacency, obs streamed out in API layout with 16-byte stores.
//   reset_kernel<G>   masked reset + observation of the current state (reset() path).
//   assign_kernel<G>  stand-alone batched lexifair assignment.
//   pack/unpack       API-layout FmState <-> internal SoA state.
//   edge_*            policy-side edge list (process_adj) by warp ballot + prefix compaction.
//   stats_reduce      fixed-order reduction of the per-warp statistic partial sums.
#include <algorithm>

#include <cstdlib>

#include "fm_device.cuh"
#include "fm_launch.h"

namespace fm {

constexpr int THREADS = 128;   // 4 warps per CTA; no block-level barrier is used

// shared memory of one assign_kernel problem, in floats (even): n^2 doubles | n^2 uint16 | 5n + 1 ints
__host__ __device__ inline int assign_smem_floats(int n) { return (2 * n * n + ((n * n + 1) >> 1) + n + 1) & ~1; }

// =============================================================================================
// The fused step.  Reference call stack: MultiAgentGraphEnv.step (environment.py:816-877).
template <int G, bool WALLS>
__global__ void __launch_bounds__(THREADS, G == 8 ? (WALLS ? 5 : 6) : (G == 4 ? 5 : (G == 16 ? 4 : 3))) step_kernel(const __grid_constant__ DevParams p) {
  extern __shared__ __align__(16) float smem[];
  constexpr int EPW = 32 / G;
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  const int env0 = p.env_begin + (blockIdx.x * (THREADS / 32) + wib) * EPW;
  if (env0 >= p.env_end) return;                 // warp-uniform
  const int gw = env0 / EPW;                     // global warp index (statistics row)
  const int nenv = min(EPW, p.env_end - env0);
  const int el = lane / G, i = lane % G;
  const int env = env0 + el;
  const int N = p.N, O = p.O, E = p.E;
  const int W = WALLS ? p.W : 0;                 // walls: entities 2N+O .. E-1 (their own instantiation)
  const bool venv = el < nenv;
  const bool act = venv && i < N;
  const unsigned gmask = (G == 32) ? FULL : (((1u << G) - 1u) << (el * G));
  const int gl = el * G;                         // first lane of my group
  const WarpSmem s = carve(p, smem, wib, env0);
  float* ent = s.ent + (size_t)el * E * ENT_STRIDE;
  float* adj = s.adj + (size_t)el * E * E;
  float* obs = s.obs + (size_t)el * N * OBS_F;
  const size_t idx = (size_t)i * p.Bp + env;

  // ---- load state ---------------------------------------------------------------------------
  float px = 0.f, py = 0.f, vx = 0.f, vy = 0.f, pd = 0.f, dtg = -1.f, treq = -1.f, dleft = -1.f, mint = 0.f;
  int gm = 0, nac = 0, noc = 0;
  float ux = 0.f, uy = 0.f;
  if (act) {
    px = p.px[idx]; py = p.py[idx]; vx = p.vx[idx]; vy = p.vy[idx]; pd = p.pdist[idx];
    dtg = p.dtg[idx]; treq = p.treq[idx]; dleft = p.dleft[idx];
    gm = p.gm[idx]; nac = p.nac[idx]; noc = p.noc[idx];
    // action decode, environment.py:301-311: u = [a1 - a2, a3 - a4] * sensitivity (5.0)
    if (p.act_idx) {
      const int a = p.act_idx[(size_t)env * N + i];
      ux = ((a == 1) ? 1.f : 0.f) - ((a == 2) ? 1.f : 0.f);
      uy = ((a == 3) ? 1.f : 0.f) - ((a == 4) ? 1.f : 0.f);
    } else {
      const float* oh = p.act_onehot + ((size_t)env * N + i) * 5;
      ux = oh[1] - oh[2];
      uy = oh[3] - oh[4];
    }
    ux *= 5.0f; uy *= 5.0f;
    const float lxx = p.lx[idx], lyy = p.ly[idx];
    ent_write(ent + (N + i) * ENT_STRIDE, lxx, lyy, 0.f, 0.f, lxx, lyy, 1.0f);
  }
  int step = 0; uint32_t episode = 0; float dmean = 0.f, dstd = 0.f;
  if (venv) {
    step = p.step[env]; episode = (uint32_t)p.episode[env]; dmean = p.dmean[env]; dstd = p.dstd[env];
    for (int k = i; k < O; k += G) {
      const float x = p.ox[(size_t)k * p.Bp + env], y = p.oy[(size_t)k * p.Bp + env];
      ent_write(ent + (2 * N + k) * ENT_STRIDE, x, y, 0.f, 0.f, x, y, 2.0f);
    }
    for (int k = i; k < W; k += G) load_wall(p, ent, env, k);
  }
  __syncwarp();

  // ---- World.step: forces (core.py:277-316, :370-404) from the positions at step entry --------
  // (== the reference's end-of-previous-step distance cache), partners in ascending entity index.
  float cfx = 0.f, cfy = 0.f;
  for (int j = 0; j < N; ++j) {
    const float qx = __shfl_sync(FULL, px, gl + j), qy = __shfl_sync(FULL, py, gl + j);
    if (act && j != i) contact_force(p, px, py, qx, qy, cfx, cfy);
  }
  if (act) {
    for (int k = 0; k < O; ++k) {
      const float* o = ent + (2 * N + k) * ENT_STRIDE;
      contact_force(p, px, py, o[0], o[1], cfx, cfy);
    }
    // walls: first as circle entities of the pair loop (they close world.entities), then the wall forces proper
    // (core.py:317-327), both from the positions at step entry
    for (int k = 0; k < W; ++k) {
      const float* w = ent + (2 * N + O + k) * ENT_STRIDE;
      contact_force_dmin(p, 0.15f, px, py, w[0], w[1], cfx, cfy);
    }
    for (int k = 0; k < W; ++k) {
      const float* w = ent + (2 * N + O + k) * ENT_STRIDE;
      wall_force(px, py, w[7] == 0.0f, w[5], w[4], cfx, cfy);
    }
  }
  const double Fx = __dadd_rn((double)ux, (double)cfx), Fy = __dadd_rn((double)uy, (double)cfy);   // mass(1.0) * u + contact
  // ---- integrate_state (core.py:338-356), float64 so that p_dist keeps its low bits for the
  // ill-conditioned mean/std fairness ratio; state is stored rounded to fp32.
  double v64x, v64y, sx, sy, pd64;
  integrate64(p, vx, vy, Fx, Fy, pd, v64x, v64y, sx, sy, pd64);
  const float npx0 = (float)__dadd_rn((double)px, sx), npy0 = (float)__dadd_rn((double)py, sy);
  float npx = npx0, npy = npy0;
  float nvx = (float)v64x, nvy = (float)v64y;
  float npd = (float)pd64;
  const int nstep = step + 1;                    // environment.py:819, :823
  if (act) {
    const float* g = ent + (N + gm) * ENT_STRIDE;
    ent_write(ent + i * ENT_STRIDE, npx, npy, nvx, nvy, g[0], g[1], 0.0f);
  }
  __syncwarp();

  // ---- calculate_distances (core.py:204-228) at the new positions -----------------------------
  double dgoal; int ncoll; bool ocoll;
  if (venv) distance_tile<G, WALLS>(p, ent, adj, env, false, i, act, gm, dgoal, ncoll, ocoll);
  else { dgoal = 0.0; ncoll = 0; ocoll = false; }
  if (act) {
    for (int k = 0; k < W; ++k) {                // is_obstacle_collision also tests the wall boxes (:670-683)
      const float* w = ent + (2 * N + O + k) * ENT_STRIDE;
      ocoll = ocoll || in_wall_box(npx, npy, w[7] == 0.0f, w[5], w[4]);
    }
  }

  // ---- per-agent loop of MultiAgentGraphEnv.step (environment.py:832-864): agent i's observation
  // and reward read world.dist_traveled_mean/stddev as left by agent i-1's info_callback
  // (navigation_graph.py:617-618), agent 0 reads last step's values.  dists_to_goal after agent j's
  // info_callback is p_dist_j unless it latched in an earlier step (:587-598).
  const bool latched = treq != -1.0f;
  const double dtg_prev = (double)dtg;
  const double dtg_new = latched ? dtg_prev : pd64;
  const bool reached = dgoal < p.min_dist_thresh;
  const double treq_prev = (double)treq;
  const double treq_new = (!latched && reached) ? (double)nstep * p.dt : treq_prev;   // :588
  const float dleft_new = latched ? dleft : (float)dgoal;
  double sum_p = 0.0, sum_v = 0.0, sum_a = 0.0;
  for (int j = 0; j < N; ++j) {
    const double pj = __shfl_sync(FULL, pd64, gl + j);
    const double aj = __shfl_sync(FULL, dtg_new, gl + j);
    const double bj = __shfl_sync(FULL, dtg_prev, gl + j);
    sum_p = __dadd_rn(sum_p, pj); sum_a = __dadd_rn(sum_a, aj); sum_v = __dadd_rn(sum_v, (j < i) ? aj : bj);
  }
  const double inv_n = 1.0 / N;
  const double mean_p = __dmul_rn(sum_p, inv_n), mean_v = __dmul_rn(sum_v, inv_n), mean_a = __dmul_rn(sum_a, inv_n);
  double q_p = 0.0, q_v = 0.0, q_a = 0.0;
  for (int j = 0; j < N; ++j) {
    const double pj = __shfl_sync(FULL, pd64, gl + j);
    const double aj = __shfl_sync(FULL, dtg_new, gl + j);
    const double bj = __shfl_sync(FULL, dtg_prev, gl + j);
    const double dp = __dsub_rn(pj, mean_p), da = __dsub_rn(aj, mean_a), dv = __dsub_rn((j < i) ? aj : bj, mean_v);
    q_p = sq_acc(q_p, dp); q_a = sq_acc(q_a, da); q_v = sq_acc(q_v, dv);
  }
  // navigation_graph.py:764-769 / :849-853.  One float64 root and one quotient per lane: the (mean, squared deviations) pair
  // the lane's fairness value comes from is selected first (first step of the episode: the travelled distances; agent 0:
  // last step's statistics from the state; agent i >= 1: the set left by agent i - 1's info_callback).
  const bool from_state = dtg != -1.0f && i == 0;
  const double mean_sel = dtg == -1.0f ? mean_p : mean_v, q_sel = dtg == -1.0f ? q_p : q_v;
  const float fparam = from_state ? ratio_eps((double)dmean, (double)dstd) : ratio_eps(mean_sel, std_from_q(q_sel, inv_n));
  const float std_a = (i == 0) ? (float)std_from_q(q_a, inv_n) : 0.0f;   // written to the state by the group's first lane only

  // reward (navigation_graph.py:760-824)
  float rew = reached ? p.goal_rew : -(float)dgoal;
  rew -= p.coll_rew * (float)ncoll;
  if (ocoll) rew -= p.coll_rew;
  if (p.fairness_reward) {
    float fair = p.fair_rew * tanhf(fparam - p.zeroshift_f);
    if (fair < -2.0f) fair = -2.0f;
    rew += fair;
  }
  rew = fminf(fmaxf(rew, p.clip_lo), p.clip_hi);
  const float own_rew = rew;
  if (p.collaborative) {                         // environment.py:866-870
    float tot = 0.f;
    for (int j = 0; j < N; ++j) tot += __shfl_sync(FULL, own_rew, gl + j);
    rew = tot;
  }
  nac += ncoll;                                  // :604-613
  noc += ocoll ? 1 : 0;                          // :602-603
  const bool done = nstep >= p.episode_length;   // environment.py:237-247 (agent.status is never set)
  const bool do_reset = venv && done && (p.auto_reset != 0);

  // ---- info rows (navigation_graph.py:625-647); world-level means as seen right after agent i's own
  // info_callback, i.e. over [new_0..new_i, prev_i+1..prev_N-1].
  const bool want_info = venv && (p.o_info != nullptr || p.stats != nullptr) && (done || p.info_every_step);
  float info[INFO_F];
  if (__any_sync(FULL, want_info)) {
    double sd = 0.0, st = 0.0;
    for (int j = 0; j < N; ++j) {
      const double aj = __shfl_sync(FULL, dtg_new, gl + j), bj = __shfl_sync(FULL, dtg_prev, gl + j);
      const double tj = __shfl_sync(FULL, treq_new, gl + j), uj = __shfl_sync(FULL, treq_prev, gl + j);
      sd = __dadd_rn(sd, (j <= i) ? aj : bj); st = __dadd_rn(st, (j <= i) ? tj : uj);
    }
    const double md = __dmul_rn(sd, inv_n), mt = __dmul_rn(st, inv_n);
    double qd = 0.0, qt = 0.0;
    for (int j = 0; j < N; ++j) {
      const double aj = __shfl_sync(FULL, dtg_new, gl + j), bj = __shfl_sync(FULL, dtg_prev, gl + j);
      const double tj = __shfl_sync(FULL, treq_new, gl + j), uj = __shfl_sync(FULL, treq_prev, gl + j);
      const double dd = __dsub_rn((j <= i) ? aj : bj, md), dtt = __dsub_rn((j <= i) ? tj : uj, mt);
      qd = sq_acc(qd, dd); qt = sq_acc(qt, dtt);
    }
    const double sdv = std_from_q(qd, inv_n), stv = std_from_q(qt, inv_n);
    double tacc = 0.0;                           // entity.state.time += dt per step (core.py:355)
    for (int k = 0; k < nstep; ++k) tacc += p.dt;
    info[0] = own_rew; info[1] = dleft_new; info[2] = (float)treq_new; info[3] = (float)nac; info[4] = (float)noc;
    info[5] = (float)md; info[6] = (float)sdv; info[7] = ratio_eps(md, sdv); info[8] = (float)dtg_new;
    info[9] = (float)tacc; info[10] = (float)mt; info[11] = (float)stv; info[12] = ratio_eps(mt, stv);
    info[13] = mint = act ? p.mintime[idx] : 0.f;
    if (act && want_info && p.o_info) {
      float* o = p.o_info + ((size_t)env * N + i) * INFO_F;
#pragma unroll
      for (int k = 0; k < INFO_F; ++k) o[k] = info[k];
    }
  } else {
#pragma unroll
    for (int k = 0; k < INFO_F; ++k) info[k] = 0.f;
  }

  // ---- episode statistics: per-warp partial sums (one row per warp, so the order of the adds is fixed) ----
  if (p.stats) {
    double* row = p.stats + (size_t)gw * (15 * N + 2);
    double r = act ? (double)rew : 0.0;
    for (int off = G; off < 32; off <<= 1) r += __shfl_xor_sync(FULL, r, off);
    if (el == 0 && i < N) atomicAdd(row + i, r);                    // RED: one add per (row, step), order fixed
    const bool term = venv && done;
    if (__any_sync(FULL, term)) {
#pragma unroll
      for (int k = 0; k < INFO_F; ++k) {
        double v = (act && done) ? (double)info[k] : 0.0;
        for (int off = G; off < 32; off <<= 1) v += __shfl_xor_sync(FULL, v, off);
        if (el == 0 && i < N) atomicAdd(row + N + i * INFO_F + k, v);
      }
    }
    const unsigned termb = __ballot_sync(FULL, term && i == 0);
    if (lane == 0) { atomicAdd(row + 15 * N, (double)__popc(termb)); atomicAdd(row + 15 * N + 1, (double)nenv); }
  }

  // ---- write back state; observation row --------------------------------------------------------
  float fobs = (float)fparam;
  float ndtg = (float)dtg_new, ntreq = (float)treq_new, ndleft = dleft_new;
  float ndmean = (float)mean_a, ndstd = std_a;            // after the last agent's info_callback
  int nstep_store = nstep;
  uint32_t nepisode = episode;
  if (__any_sync(FULL, do_reset)) {
    // graphworker auto-reset (env_wrappers.py:859-865): obs / node_obs / adj come from the new
    // episode; reward / done / info stay terminal.
    __syncwarp();          // the entity table is rewritten below: every lane is past its distance_tile reads (racecheck)
    float rx = npx, ry = npy, rmint = act ? p.mintime[idx] : 0.f;
    int rgm = gm;
    // An entry of the pending block generated for this env's episode key (prefetch_kernel) replaces the rejection
    // sampling and the lexifair solve: same Philox stream, same bits.
    bool use_pend = false;
    if (do_reset && p.q_tag != nullptr) {            // acquire: the entry's data is visible once its tag is
      int tag;
      asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(tag) : "l"(p.q_tag + env) : "memory");
      use_pend = tag == (int)episode;
    }
    if (__any_sync(FULL, use_pend)) {
      int pgm = 0;
      if (use_pend) {
        if (i < N) {
          rx = p.q_px[idx]; ry = p.q_py[idx]; pgm = p.q_gm[idx];
          const float lxx = p.q_lx[idx], lyy = p.q_ly[idx];
          ent_write(ent + (N + i) * ENT_STRIDE, lxx, lyy, 0.f, 0.f, lxx, lyy, 1.0f);
          p.lx[idx] = lxx; p.ly[idx] = lyy;
        }
        for (int k = i; k < O; k += G) {
          const float x = p.q_ox[(size_t)k * p.Bp + env], y = p.q_oy[(size_t)k * p.Bp + env];
          ent_write(ent + (2 * N + k) * ENT_STRIDE, x, y, 0.f, 0.f, x, y, 2.0f);
          p.ox[(size_t)k * p.Bp + env] = x; p.oy[(size_t)k * p.Bp + env] = y;
        }
        for (int k = i; k < W; k += G) {
          const size_t wi = (size_t)k * p.Bp + env;
          p.wax[wi] = p.q_wax[wi]; p.wor[wi] = p.q_wor[wi];
          store_wall(ent, N, O, k, p.q_wax[wi], p.q_wor[wi], p.wlen[env]);
        }
      }
      __syncwarp();
      if (use_pend && i < N) {
        const float* og = ent + (N + gm) * ENT_STRIDE;     // min_time with the previous episode's goal_match (:545-547)
        if (p.has_max_speed) rmint = (float)(dist64(rx, ry, og[0], og[1]) / p.max_speed);
        rgm = pgm;
        const float* g = ent + (N + rgm) * ENT_STRIDE;
        ent_write(ent + i * ENT_STRIDE, rx, ry, 0.f, 0.f, g[0], g[1], 0.0f);
      }
      __syncwarp();
    }
    if (__any_sync(FULL, do_reset && !use_pend))
      reset_group<G, WALLS>(p, s, el, i, env, do_reset && !use_pend, gmask, episode, rgm, rx, ry, rmint, p.lx, p.ly, p.ox, p.oy, p.wax, p.wor, true);
    if (do_reset) {
      gm = rgm; npx = rx; npy = ry; nvx = 0.f; nvy = 0.f; npd = 0.f;
      ndtg = -1.f; ntreq = -1.f; ndleft = -1.f; nac = 0; noc = 0; nstep_store = 0; nepisode = episode + 1;
      fobs = 0.f;                                // mean(p_dist = 0) / (std + 1e-4)
      if (act) p.mintime[idx] = rmint;
      double d2; int c2; bool o2;
      distance_tile<G, WALLS>(p, ent, adj, env, true, i, act, gm, d2, c2, o2);
    }
  }
  if (act) {
    p.px[idx] = npx; p.py[idx] = npy; p.vx[idx] = nvx; p.vy[idx] = nvy; p.pdist[idx] = npd;
    p.dtg[idx] = ndtg; p.treq[idx] = ntreq; p.dleft[idx] = ndleft;
    p.gm[idx] = gm; p.nac[idx] = nac; p.noc[idx] = noc;
    const float gx = ent[i * ENT_STRIDE + 4], gy = ent[i * ENT_STRIDE + 5];
    obs[i * OBS_F + 0] = nvx; obs[i * OBS_F + 1] = nvy; obs[i * OBS_F + 2] = npx; obs[i * OBS_F + 3] = npy;
    obs[i * OBS_F + 4] = gx - npx; obs[i * OBS_F + 5] = gy - npy; obs[i * OBS_F + 6] = fobs;
    if (p.o_rew) p.o_rew[(size_t)env * N + i] = rew;
    if (p.o_done) p.o_done[(size_t)env * N + i] = done ? 1 : 0;
  }
  if (venv && i == 0) {
    p.step[env] = nstep_store; p.episode[env] = (int)nepisode; p.dmean[env] = ndmean; p.dstd[env] = ndstd;
  }
  __syncwarp();
  emit_tiles<WALLS>(p, s, env0, nenv, lane);
}

// =============================================================================================
// reset() / observe: GraphSubprocVecEnv.reset -> MultiAgentGraphEnv.reset (environment.py:882-898).
template <int G, bool WALLS>
__global__ void __launch_bounds__(THREADS) reset_kernel(const __grid_constant__ DevParams p) {
  extern __shared__ __align__(16) float smem[];
  constexpr int EPW = 32 / G;
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  const int env0 = p.env_begin + (blockIdx.x * (THREADS / 32) + wib) * EPW;
  if (env0 >= p.env_end) return;
  const int nenv = min(EPW, p.env_end - env0);
  const int el = lane / G, i = lane % G;
  const int env = env0 + el;
  const int N = p.N, O = p.O, E = p.E;
  const int W = WALLS ? p.W : 0;                 // walls: entities 2N+O .. E-1 (their own instantiation)
  const bool venv = el < nenv;
  const bool act = venv && i < N;
  const unsigned gmask = (G == 32) ? FULL : (((1u << G) - 1u) << (el * G));
  const int gl = el * G;
  const WarpSmem s = carve(p, smem, wib, env0);
  float* ent = s.ent + (size_t)el * E * ENT_STRIDE;
  float* adj = s.adj + (size_t)el * E * E;
  float* obs = s.obs + (size_t)el * N * OBS_F;
  const size_t idx = (size_t)i * p.Bp + env;

  float px = 0.f, py = 0.f, vx = 0.f, vy = 0.f, pd = 0.f, dtg = -1.f, mint = 0.f;
  int gm = 0;
  if (act) {
    px = p.px[idx]; py = p.py[idx]; vx = p.vx[idx]; vy = p.vy[idx]; pd = p.pdist[idx]; dtg = p.dtg[idx];
    gm = p.gm[idx]; mint = p.mintime[idx];
    const float lxx = p.lx[idx], lyy = p.ly[idx];
    ent_write(ent + (N + i) * ENT_STRIDE, lxx, lyy, 0.f, 0.f, lxx, lyy, 1.0f);
  }
  uint32_t episode = 0; float dmean = 0.f, dstd = 0.f;
  bool do_reset = false;
  if (venv) {
    episode = (uint32_t)p.episode[env]; dmean = p.dmean[env]; dstd = p.dstd[env];
    do_reset = p.observe_only ? false : (p.reset_mask ? (p.reset_mask[env] != 0) : true);
    for (int k = i; k < O; k += G) {
      const float x = p.ox[(size_t)k * p.Bp + env], y = p.oy[(size_t)k * p.Bp + env];
      ent_write(ent + (2 * N + k) * ENT_STRIDE, x, y, 0.f, 0.f, x, y, 2.0f);
    }
    for (int k = i; k < W; k += G) load_wall(p, ent, env, k);
  }
  __syncwarp();
  if (act) {
    const float* g = ent + (N + gm) * ENT_STRIDE;
    ent_write(ent + i * ENT_STRIDE, px, py, vx, vy, g[0], g[1], 0.0f);
  }
  __syncwarp();
  if (__any_sync(FULL, do_reset)) {
    reset_group<G, WALLS>(p, s, el, i, env, do_reset, gmask, episode, gm, px, py, mint, p.lx, p.ly, p.ox, p.oy, p.wax, p.wor, true);
    if (do_reset && act) {
      vx = 0.f; vy = 0.f; pd = 0.f; dtg = -1.f;
      p.px[idx] = px; p.py[idx] = py; p.vx[idx] = 0.f; p.vy[idx] = 0.f; p.pdist[idx] = 0.f;
      p.dtg[idx] = -1.f; p.treq[idx] = -1.f; p.dleft[idx] = -1.f;
      p.gm[idx] = gm; p.nac[idx] = 0; p.noc[idx] = 0; p.mintime[idx] = mint;
    }
    if (do_reset && i == 0) { p.step[env] = 0; p.episode[env] = (int)(episode + 1); }
  }
  // observation() on the current state (navigation_graph.py:826-857)
  double sum_p = 0.0;
  const double pd64 = (double)pd;
  for (int j = 0; j < N; ++j) sum_p = __dadd_rn(sum_p, __shfl_sync(FULL, pd64, gl + j));
  const double inv_n = 1.0 / N;
  const double mean_p = __dmul_rn(sum_p, inv_n);
  double q_p = 0.0;
  for (int j = 0; j < N; ++j) { const double d = __dsub_rn(__shfl_sync(FULL, pd64, gl + j), mean_p); q_p = sq_acc(q_p, d); }
  const double std_p = std_from_q(q_p, inv_n);
  const float fparam = (dtg == -1.0f) ? ratio_eps(mean_p, std_p) : ratio_eps((double)dmean, (double)dstd);
  double dgoal; int ncoll; bool ocoll;
  if (venv) distance_tile<G, WALLS>(p, ent, adj, env, do_reset, i, act, gm, dgoal, ncoll, ocoll);
  if (act) {
    const float gx = ent[i * ENT_STRIDE + 4], gy = ent[i * ENT_STRIDE + 5];
    obs[i * OBS_F + 0] = vx; obs[i * OBS_F + 1] = vy; obs[i * OBS_F + 2] = px; obs[i * OBS_F + 3] = py;
    obs[i * OBS_F + 4] = gx - px; obs[i * OBS_F + 5] = gy - py; obs[i * OBS_F + 6] = (float)fparam;
  }
  __syncwarp();
  emit_tiles<WALLS>(p, s, env0, nenv, lane);
}

// =============================================================================================
// Placement + lexifair assignment of every env's NEXT episode, ahead of time (navigation_graph.py:264-570; the draws
// depend only on (seed, global env, episode key)).  Launched on a side stream right after the kernel that advanced
// the episode counters; it overlaps the memory-bound regular steps of the episode, and the terminal step copies the
// entry (step_kernel, `use_pend`).  Envs whose entry already carries the current key are skipped.
template <int G, bool WALLS>
__global__ void __launch_bounds__(THREADS) prefetch_kernel(const __grid_constant__ DevParams p) {
  extern __shared__ __align__(16) float smem[];
  constexpr int EPW = 32 / G;
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  const int env0 = p.env_begin + (blockIdx.x * (THREADS / 32) + wib) * EPW;
  if (env0 >= p.env_end) return;
  const int nenv = min(EPW, p.env_end - env0);
  const int el = lane / G, i = lane % G;
  const int env = env0 + el;
  const bool venv = el < nenv;
  const unsigned gmask = (G == 32) ? FULL : (((1u << G) - 1u) << (el * G));
  const WarpSmem s = carve_prefetch(p, smem, wib);
  const uint32_t episode = venv ? (uint32_t)p.episode[env] : 0u;
  const bool need = venv && p.q_tag[env] != (int)episode;
  if (!__any_sync(FULL, need)) return;
  int gm = 0;
  float x = 0.f, y = 0.f, mint = 0.f;
  reset_group<G, WALLS>(p, s, el, i, env, need, gmask, episode, gm, x, y, mint, p.q_lx, p.q_ly, p.q_ox, p.q_oy, p.q_wax, p.q_wor, false);
  if (need && i < p.N) {
    const size_t idx = (size_t)i * p.Bp + env;
    p.q_px[idx] = x; p.q_py[idx] = y; p.q_gm[idx] = gm;
  }
  __syncwarp();
  if (need && i == 0) {                              // the entry is complete (every lane's stores, ordered by the warp barrier) before its tag
    __threadfence();
    asm volatile("st.release.gpu.global.s32 [%0], %1;" :: "l"(p.q_tag + env), "r"((int)episode) : "memory");
  }
}

// =============================================================================================
// Stand-alone batched lexifair (marl_fair_assign.py:16-55).  A NaN or +-inf cost (or coordinate: dist64 alone would turn a
// NaN into a distance of 0) breaks the total order the sort relies on, so such a problem gets -1 in every entry of its row
// instead of an arbitrary permutation; the other problems of the batch are unaffected.  The check lives here, not in
// lexifair_group, whose other callers (resets, prefetch) solve distances of finite positions.
template <int G>
__global__ void __launch_bounds__(THREADS) assign_kernel(const double* __restrict__ costs, const float* __restrict__ apos,
                                                         const float* __restrict__ gpos, int num, int n, int* __restrict__ out) {
  extern __shared__ __align__(16) float smem[];
  constexpr int EPW = 32 / G;
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  const int gw = blockIdx.x * (THREADS / 32) + wib;
  const int el = lane / G, i = lane % G;
  const int prob = gw * EPW + el;
  const unsigned gmask = (G == 32) ? FULL : (((1u << G) - 1u) << (el * G));
  const int per_group = assign_smem_floats(n);                   // cost (doubles) | sort permutation (uint16) | int scratch
  float* base = smem + (size_t)(wib * EPW + el) * per_group;
  double* cost = reinterpret_cast<double*>(base);
  uint16_t* ord = reinterpret_cast<uint16_t*>(base + 2 * n * n);
  int* asg = reinterpret_cast<int*>(base + 2 * n * n + ((n * n + 1) >> 1));
  if (prob >= num) return;                                        // group-uniform; only group syncs below
  bool finite = true;
  if (i < n) {
    for (int j = 0; j < n; ++j) {
      if (costs) {
        const double c = costs[((size_t)prob * n + i) * n + j];
        finite = finite && isfinite(c);
        cost[i * n + j] = c;
      } else {                                                    // dist64 in two halves: a NaN coordinate stays NaN in
        const float* a = apos + ((size_t)prob * n + i) * 2;       // the square, its root would make it 0
        const float* g = gpos + ((size_t)prob * n + j) * 2;
        const double q = dist64_sq(a[0], a[1], g[0], g[1]);
        finite = finite && isfinite(q);
        cost[i * n + j] = dsqrt_fast(q);
      }
    }
  }
  if (!__all_sync(gmask, finite)) {
    if (i < n) out[(size_t)prob * n + i] = -1;
    return;
  }
  __syncwarp(gmask);
  const int g = lexifair_group<G>(cost, ord, asg, n, i, gmask);
  if (i < n) out[(size_t)prob * n + i] = g;
}

// =============================================================================================
// FmState (API layout) <-> internal SoA.  One thread per (env, slot), slot < max(N, O).
__global__ void state_io_kernel(const DevParams p, const HostState st, int to_internal) {
  const int S = max(p.N, max(max(p.O, p.W), 1));
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)p.B * S) return;
  const int env = (int)(t / S), k = (int)(t % S);
  const int N = p.N, O = p.O;
  const size_t si = (size_t)k * p.Bp + env;
  if (k < N) {
    const size_t ai = (size_t)env * N + k;
#define FM_IO_F(ptr, arr, stride, comp) \
  if (st.ptr) { if (to_internal) p.arr[si] = st.ptr[ai * stride + comp]; else st.ptr[ai * stride + comp] = p.arr[si]; }
    FM_IO_F(pos, px, 2, 0) FM_IO_F(pos, py, 2, 1) FM_IO_F(vel, vx, 2, 0) FM_IO_F(vel, vy, 2, 1)
    FM_IO_F(p_dist, pdist, 1, 0) FM_IO_F(landmark_pos, lx, 2, 0) FM_IO_F(landmark_pos, ly, 2, 1)
    FM_IO_F(goal_match, gm, 1, 0) FM_IO_F(dists_to_goal, dtg, 1, 0) FM_IO_F(times_required, treq, 1, 0)
    FM_IO_F(dist_left_to_goal, dleft, 1, 0) FM_IO_F(num_agent_collisions, nac, 1, 0)
    FM_IO_F(num_obstacle_collisions, noc, 1, 0) FM_IO_F(min_time, mintime, 1, 0)
#undef FM_IO_F
  }
  if (k < O && st.obstacle_pos) {
    const size_t oi = ((size_t)env * O + k) * 2;
    if (to_internal) { p.ox[si] = st.obstacle_pos[oi]; p.oy[si] = st.obstacle_pos[oi + 1]; }
    else { st.obstacle_pos[oi] = p.ox[si]; st.obstacle_pos[oi + 1] = p.oy[si]; }
  }
  if (k < p.W) {
    const size_t wi = (size_t)env * p.W + k;
    if (st.wall_axis) { if (to_internal) p.wax[si] = st.wall_axis[wi]; else st.wall_axis[wi] = p.wax[si]; }
    if (st.wall_orient) { if (to_internal) p.wor[si] = st.wall_orient[wi]; else st.wall_orient[wi] = p.wor[si]; }
  }
  if (k == 0 && st.wall_len && p.W > 0) { if (to_internal) p.wlen[env] = st.wall_len[env]; else st.wall_len[env] = p.wlen[env]; }
  if (k == 0) {
#define FM_IO_E(ptr, arr) \
  if (st.ptr) { if (to_internal) p.arr[env] = st.ptr[env]; else st.ptr[env] = p.arr[env]; }
    FM_IO_E(dist_traveled_mean, dmean) FM_IO_E(dist_traveled_stddev, dstd) FM_IO_E(step, step) FM_IO_E(episode, episode)
#undef FM_IO_E
  }
}

// make_world defaults (navigation_graph.py:93, :137-138): goal_match = arange(N), latches = -1.
__global__ void state_init_kernel(const DevParams p) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)p.Bp * p.N) return;
  const int k = (int)(t / p.Bp);
  p.gm[t] = k; p.dtg[t] = -1.f; p.treq[t] = -1.f; p.dleft[t] = -1.f;
  p.mintime[t] = __int_as_float(0x7f800000);   // agent.goal_min_time = np.inf (core.py:127)
  if (k == 0 && p.W > 0) {                       // scenario.wall_length = U(0.2, 0.8) * world_size / 4, once per env (:183-185)
    const int env = (int)(t % p.Bp);
    float u0, u1;
    draw_u01(p, p.env_offset + env, 0xffffffffu, 0u, u0, u1);
    p.wlen[env] = __fmul_rn(__fadd_rn(0.2f, __fmul_rn(0.6f, u0)), p.world_size * 0.25f);
  }
}

// =============================================================================================
// Edge list (gnn_new.py:381-413).  One warp per graph.
__device__ __forceinline__ bool edge_pred(float d, float thr, int inclusive) {
  return (inclusive ? (d <= thr) : (d < thr)) && (d > 0.0f);
}

constexpr int EDGE_WPB = 8;          // graphs (warps) per CTA of the edge-list kernels

// Pass 1: edges per graph (one warp per graph) and per CTA.
__global__ void edge_count_kernel(const float* __restrict__ adj, int num_graphs, int EE, float thr, int inclusive,
                                  int* __restrict__ counts, long long* __restrict__ blocksums) {
  __shared__ int wc[EDGE_WPB];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int g = blockIdx.x * EDGE_WPB + w;
  int c = 0;
  if (g < num_graphs) {
    const float* a = adj + (size_t)g * EE;
#pragma unroll 8
    for (int q = lane; q < EE; q += 32) c += edge_pred(__ldg(a + q), thr, inclusive) ? 1 : 0;
    for (int off = 16; off > 0; off >>= 1) c += __shfl_xor_sync(FULL, c, off);
    if (lane == 0) counts[g] = c;
  }
  if (lane == 0) wc[w] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
#pragma unroll
    for (int k = 0; k < EDGE_WPB; ++k) t += wc[k];
    blocksums[blockIdx.x] = t;
  }
}

// Pass 2: exclusive scan of the per-CTA sums by ONE block of 32 warps, in place, scaled by `repeat`.  Warp w owns the
// contiguous segment [w * seg, (w + 1) * seg) and walks it 32 entries at a time (coalesced loads, shuffle scan, running
// carry); the 32 segment totals are scanned by warp 0 and added in a second coalesced sweep.  num_blocks = num_graphs
// / 8: 32 K entries at 262 144 graphs.  Also writes the end sentinel of graph_offsets and nnz.
__global__ void edge_scan_kernel(long long* __restrict__ blocksums, int num_blocks, int repeat, long long* __restrict__ sentinel,
                                 long long* __restrict__ nnz_out) {
  __shared__ long long wtot[32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int seg = ((num_blocks + 31) / 32 + 31) & ~31;              // per-warp segment, a multiple of 32 entries
  const int lo = min(num_blocks, w * seg), hi = min(num_blocks, lo + seg);
  long long carry = 0;
  for (int k0 = lo; k0 < hi; k0 += 32) {
    const int k = k0 + lane;
    const long long c = (k < hi) ? blocksums[k] : 0;
    long long incl = c;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) { const long long o = __shfl_up_sync(FULL, incl, off); if (lane >= off) incl += o; }
    if (k < hi) blocksums[k] = carry + incl - c;                    // exclusive prefix inside the segment
    carry += __shfl_sync(FULL, incl, 31);
  }
  if (lane == 0) wtot[w] = carry;
  __syncthreads();
  if (w == 0) {
    const long long t = wtot[lane];
    long long incl = t;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) { const long long o = __shfl_up_sync(FULL, incl, off); if (lane >= off) incl += o; }
    wtot[lane] = incl - t;                                           // exclusive prefix of the segment totals
    if (lane == 31) { *sentinel = incl * repeat; if (nnz_out) *nnz_out = incl * repeat; }
  }
  __syncthreads();
  const long long base = wtot[w];
  for (int k = lo + lane; k < hi; k += 32) blocksums[k] = (blocksums[k] + base) * repeat;
}

// Pass 3: graph offsets inside the CTA from the 8 counts, then ballot + popc compaction in (b, i, j) order.
__global__ void __launch_bounds__(EDGE_WPB * 32, 6)   // <= 40 registers: 48 warps / SM (the unrolled compaction wanted 96 -> 16 warps; same-box A/B: edge stage 0.70 -> 0.49 ms at config 3)
edge_emit_kernel(const float* __restrict__ adj, int num_graphs, int E, float thr, int inclusive, int repeat,
                                 long long capacity, const int* __restrict__ counts, const long long* __restrict__ blockoffs,
                                 long long* __restrict__ graph_offsets, long long* __restrict__ edge_index,
                                 float* __restrict__ edge_attr) {
  __shared__ int wc[EDGE_WPB];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int g = blockIdx.x * EDGE_WPB + w;
  const int cnt = (g < num_graphs) ? counts[g] : 0;
  if (lane == 0) wc[w] = cnt;
  __syncthreads();
  if (g >= num_graphs) return;
  int before = 0;
#pragma unroll
  for (int k = 0; k < EDGE_WPB; ++k) before += (k < w) ? wc[k] : 0;
  const long long base0 = blockoffs[blockIdx.x] + (long long)before * repeat;
  if (lane < repeat) graph_offsets[(size_t)g * repeat + lane] = base0 + (long long)lane * cnt;
  for (int cp = 32 + lane; cp < repeat; cp += 32) graph_offsets[(size_t)g * repeat + cp] = base0 + (long long)cp * cnt;
  const int EE = E * E;
  const float* a = adj + (size_t)g * EE;
  const unsigned magic = (E <= 100) ? ((1u << 20) + E - 1) / E : 0u;       // q / E == (q * magic) >> 20 for q < 2^20 / E
  int run = 0;
  constexpr int U = 8;                               // 8 independent loads in flight per lane before the compaction
  for (int q0 = 0; q0 < EE; q0 += 32 * U) {
    float dv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) { const int q = q0 + u * 32 + lane; dv[u] = (q < EE) ? __ldg(a + q) : 0.0f; }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int q = q0 + u * 32 + lane;
      if (q0 + u * 32 >= EE) break;                  // warp-uniform
      const float d = dv[u];
      const bool pr = (q < EE) && edge_pred(d, thr, inclusive);
      const unsigned b = __ballot_sync(FULL, pr);
      if (pr) {
        const int k = run + __popc(b & ((1u << lane) - 1u));
        const int r = magic ? (int)(((unsigned)q * magic) >> 20) : q / E;
        const int c = q - r * E;
        for (int cp = 0; cp < repeat; ++cp) {
          const long long pos = base0 + (long long)cp * cnt + k;
          if (pos < capacity) {
            const long long node0 = ((long long)g * repeat + cp) * E;
            __stcs(edge_index + pos, node0 + r);
            __stcs(edge_index + capacity + pos, node0 + c);
            __stcs(edge_attr + pos, d);
          }
        }
      }
      run += __popc(b);
    }
  }
}

// =============================================================================================
// One block per statistic: fixed thread -> row mapping and a fixed-shape tree, so the result does
// not depend on scheduling (deterministic for a given launch geometry).
__global__ void stats_reduce_kernel(double* __restrict__ partial, int rows, int K, double* __restrict__ out, int clear) {
  __shared__ double sh[256];
  const int k = blockIdx.x;
  double acc = 0.0;
  for (int r = threadIdx.x; r < rows; r += 256) {
    acc += partial[(size_t)r * K + k];
    if (clear) partial[(size_t)r * K + k] = 0.0;
  }
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int off = 128; off > 0; off >>= 1) {
    if ((int)threadIdx.x < off) sh[threadIdx.x] += sh[threadIdx.x + off];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[k] = sh[0];
}

// =============================================================================================
// Launchers (host side of this translation unit).
template <int G, bool WALLS>
static cudaError_t launch_step_g(const DevParams& p, cudaStream_t st, bool is_reset) {
  constexpr int EPW = 32 / G;
  const int warps = (p.env_end - p.env_begin + EPW - 1) / EPW;
  const int blocks = (warps + THREADS / 32 - 1) / (THREADS / 32);
  if (blocks <= 0) return cudaSuccess;
  const size_t smem = (size_t)p.sm_per_warp * (THREADS / 32) * sizeof(float);
  if (is_reset) reset_kernel<G, WALLS><<<blocks, THREADS, smem, st>>>(p);
  else step_kernel<G, WALLS><<<blocks, THREADS, smem, st>>>(p);
  return cudaGetLastError();
}

template <int G, bool WALLS>
static cudaError_t launch_prefetch_g(const DevParams& p, cudaStream_t st) {
  constexpr int EPW = 32 / G;
  const int warps = (p.env_end - p.env_begin + EPW - 1) / EPW;
  const int blocks = (warps + THREADS / 32 - 1) / (THREADS / 32);
  if (blocks <= 0) return cudaSuccess;
  const size_t smem = (size_t)p.sm_pf_per_warp * (THREADS / 32) * sizeof(float);
  prefetch_kernel<G, WALLS><<<blocks, THREADS, smem, st>>>(p);
  return cudaGetLastError();
}

// group size x walls -> instantiation (the wall terms live in their own kernels: the wall-free ones keep their
// register budgets, e.g. 80 at G = 8)
#define FM_DISPATCH_G(fn, ...)                                                              \
  switch (group_size(p.N)) {                                                                \
    case 4: return p.W > 0 ? fn<4, true>(__VA_ARGS__) : fn<4, false>(__VA_ARGS__);          \
    case 8: return p.W > 0 ? fn<8, true>(__VA_ARGS__) : fn<8, false>(__VA_ARGS__);          \
    case 16: return p.W > 0 ? fn<16, true>(__VA_ARGS__) : fn<16, false>(__VA_ARGS__);       \
    default: return p.W > 0 ? fn<32, true>(__VA_ARGS__) : fn<32, false>(__VA_ARGS__);       \
  }

cudaError_t launch_prefetch(const DevParams& p, cudaStream_t st) { FM_DISPATCH_G(launch_prefetch_g, p, st) }

template <int G, bool WALLS>
static cudaError_t prepare_g(const DevParams& p) {
  const int smem = p.sm_per_warp * (THREADS / 32) * (int)sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(reset_kernel<G, WALLS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(prefetch_kernel<G, WALLS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           p.sm_pf_per_warp * (THREADS / 32) * (int)sizeof(float));
  if (e != cudaSuccess) return e;
  if (const char* v = getenv("FM_CARVEOUT"); v && v[0] == '1') {      // A/B: largest shared-memory carve-out instead of the driver's pick
    e = cudaFuncSetAttribute(step_kernel<G, WALLS>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
  }
  return cudaFuncSetAttribute(step_kernel<G, WALLS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
}

int group_size(int n) { return n <= 4 ? 4 : (n <= 8 ? 8 : (n <= 16 ? 16 : 32)); }

int num_warps(int B, int N) { const int epw = 32 / group_size(N); return (B + epw - 1) / epw; }

cudaError_t prepare_kernels(const DevParams& p) {
  if (p.mapping == 1) {
    cudaError_t e = aw_prepare(p);
    if (e != cudaSuccess || !p.q_tag) return e;       // the agent-warp kernels consume the entries prefetch_kernel<G> produces
  }
  FM_DISPATCH_G(prepare_g, p)
}

cudaError_t launch_step(const DevParams& p, cudaStream_t st, bool is_reset) {
  if (p.mapping == 1) return aw_launch(p, st, is_reset);
  FM_DISPATCH_G(launch_step_g, p, st, is_reset)
}

template <int G>
static cudaError_t launch_assign_g(const double* costs, const float* apos, const float* gpos, int num, int n, int* out,
                                   cudaStream_t st) {
  constexpr int EPW = 32 / G;
  const int warps = (num + EPW - 1) / EPW;
  const int blocks = (warps + THREADS / 32 - 1) / (THREADS / 32);
  const int per_group = assign_smem_floats(n);
  const size_t smem = (size_t)per_group * EPW * (THREADS / 32) * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(assign_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  assign_kernel<G><<<blocks, THREADS, smem, st>>>(costs, apos, gpos, num, n, out);
  return cudaGetLastError();
}

cudaError_t launch_assign(const double* costs, const float* apos, const float* gpos, int num, int n, int* out,
                          cudaStream_t st) {
  if (num <= 0) return cudaSuccess;
  switch (group_size(n)) {
    case 4: return launch_assign_g<4>(costs, apos, gpos, num, n, out, st);
    case 8: return launch_assign_g<8>(costs, apos, gpos, num, n, out, st);
    case 16: return launch_assign_g<16>(costs, apos, gpos, num, n, out, st);
    default: return launch_assign_g<32>(costs, apos, gpos, num, n, out, st);
  }
}

cudaError_t launch_state_io(const DevParams& p, const HostState& hs, int to_internal, cudaStream_t st) {
  const int S = std::max(p.N, std::max(std::max(p.O, p.W), 1));
  const long long total = (long long)p.B * S;
  const int blocks = (int)((total + 255) / 256);
  state_io_kernel<<<blocks, 256, 0, st>>>(p, hs, to_internal);
  return cudaGetLastError();
}

cudaError_t launch_state_init(const DevParams& p, cudaStream_t st) {
  const long long total = (long long)p.Bp * p.N;
  state_init_kernel<<<(int)((total + 255) / 256), 256, 0, st>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_edge_list(const float* adj, int num_graphs, int E, float thr, int inclusive, int repeat,
                             long long capacity, int* counts, long long* blocksums, long long* graph_offsets,
                             long long* edge_index, float* edge_attr, long long* nnz_out, cudaStream_t st) {
  const int blocks = (num_graphs + EDGE_WPB - 1) / EDGE_WPB;
  if (blocks > 0) edge_count_kernel<<<blocks, EDGE_WPB * 32, 0, st>>>(adj, num_graphs, E * E, thr, inclusive, counts, blocksums);
  edge_scan_kernel<<<1, 1024, 0, st>>>(blocksums, blocks, repeat, graph_offsets + (size_t)num_graphs * repeat, nnz_out);
  if (blocks > 0)
    edge_emit_kernel<<<blocks, EDGE_WPB * 32, 0, st>>>(adj, num_graphs, E, thr, inclusive, repeat, capacity, counts, blocksums,
                                                      graph_offsets, edge_index, edge_attr);
  return cudaGetLastError();
}

int edge_list_blocks(int num_graphs) { return (num_graphs + EDGE_WPB - 1) / EDGE_WPB; }

__global__ void pair_dist_kernel(const float* __restrict__ a, const float* __restrict__ b, long long num, double* __restrict__ out) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < num) out[k] = dist64(a[2 * k], a[2 * k + 1], b[2 * k], b[2 * k + 1]);
}

cudaError_t launch_pair_dist(const float* a, const float* b, long long num, double* out, cudaStream_t st) {
  if (num <= 0) return cudaSuccess;
  pair_dist_kernel<<<(int)((num + 255) / 256), 256, 0, st>>>(a, b, num, out);
  return cudaGetLastError();
}

cudaError_t launch_stats_reduce(double* partial, int rows, int K, double* out, int clear, cudaStream_t st) {
  stats_reduce_kernel<<<K, 256, 0, st>>>(partial, rows, K, out, clear);
  return cudaGetLastError();
}

}  // namespace fm
