// C ABI of libfairmarl.so (include/fairmarl.h): handle management, argument checking, launches.
// No torch types, no exceptions across the boundary, no CPU fallback.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "fm_device.cuh"
#include "fm_launch.h"

using fm::DevParams;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

namespace fm {
int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
}  // namespace fm

#define FM_CUDA(expr)                                                                            \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) return fail(FM_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define FM_MAX_LANES 8

struct FmHandle {
  FmConfig cfg;
  int device;
  DevParams p;
  void* state_block;
  double* stats;
  int stats_rows, K;
  long long launches;
  // fm_step_many: env-range lanes on side streams, so that the partial last wave and the launch gap of
  // one range are filled by the kernels of the others (created on first use)
  cudaStream_t lane_stream[FM_MAX_LANES];
  cudaEvent_t lane_fork, lane_join[FM_MAX_LANES];
  int lanes_ready;
  // next-episode prefetch (group mapping, DESIGN.md 4.2): pending block, one side stream + events per lane, and the
  // host's view of the episode phase (all envs share one step counter after a full reset: "lockstep")
  void* pend_block;
  int pf_on, pf_ready_made, pf_used[FM_MAX_LANES];
  cudaStream_t pf_stream[FM_MAX_LANES];
  cudaEvent_t pf_go[FM_MAX_LANES], pf_ready[FM_MAX_LANES];
  int lockstep, host_step;
  // agent-warp mapping: persistent rollout kernel (fm_roll.cu).  Control block (zero between launches), one wave of CTAs.
  void* roll_ctl;
  int roll_on, roll_max_ctas, roll_stagger_ns, roll_stagger1_ns;
  int lanes_override;        // FM_LANES (diagnostic), read once at fm_create; 0 = automatic
  // device staging for the *_host entry points (allocated on first use)
  float* st_onehot;
  uint8_t* st_mask;
  FmOutputs st_out;
  bool staging;
};

static inline int round4(long long x) { return (int)((x + 3) & ~3LL); }

static int use_device(int device) {
  int cur = -1;
  FM_CUDA(cudaGetDevice(&cur));
  if (cur != device) FM_CUDA(cudaSetDevice(device));
  return FM_OK;
}

extern "C" {

int fm_abi_version(void) { return FM_ABI_VERSION; }
const char* fm_last_error(void) { return g_err; }
int fm_stats_len(int32_t n) { return 15 * n + 2; }

int fm_create(const FmConfig* cfg, int device, FmHandle** out) {
  if (!cfg || !out) return fail(FM_ERR_INVALID_ARG, "fm_create: null argument");
  *out = nullptr;
  if (cfg->num_envs <= 0) return fail(FM_ERR_INVALID_ARG, "fm_create: num_envs must be > 0 (got %d)", cfg->num_envs);
  if (cfg->num_agents < 1 || cfg->num_agents > FM_MAX_AGENTS)
    return fail(FM_ERR_INVALID_ARG, "fm_create: num_agents must be in 1..%d (got %d)", FM_MAX_AGENTS, cfg->num_agents);
  if (cfg->num_walls < 0 || cfg->num_walls > 2)
    return fail(FM_ERR_INVALID_ARG, "fm_create: num_walls must be 0, 1 or 2 (got %d)", cfg->num_walls);
  if (cfg->num_walls > 0 && cfg->graph_feat_global)
    return fail(FM_ERR_UNSUPPORTED, "fm_create: wall entities have no global features (navigation_graph.py:1074-1075)");
  if (cfg->num_walls > 0 && cfg->mapping == 2 && !fm::aw_supported(cfg->num_agents, cfg->num_obstacles, cfg->num_walls))
    return fail(FM_ERR_UNSUPPORTED, "fm_create: the agent-warp kernels are not compiled for N=%d O=%d with %d wall(s)",
                cfg->num_agents, cfg->num_obstacles, cfg->num_walls);
  if (cfg->num_obstacles < 0 || cfg->num_obstacles > 64)
    return fail(FM_ERR_INVALID_ARG, "fm_create: num_obstacles must be in 0..64 (got %d)", cfg->num_obstacles);
  if (cfg->episode_length < 1) return fail(FM_ERR_INVALID_ARG, "fm_create: episode_length must be >= 1");
  if (cfg->mapping < 0 || cfg->mapping > 2) return fail(FM_ERR_INVALID_ARG, "fm_create: mapping must be 0..2 (got %d)", cfg->mapping);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(FM_ERR_NO_DEVICE, "fm_create: no CUDA device (this library has no CPU path)");
  }
  if (device < 0 || device >= ndev) return fail(FM_ERR_INVALID_ARG, "fm_create: device %d out of range (%d devices)", device, ndev);
  int rc = use_device(device);
  if (rc) return rc;

  FmHandle* h = new (std::nothrow) FmHandle();
  if (!h) return fail(FM_ERR_CUDA, "fm_create: out of host memory");
  memset(h, 0, sizeof(*h));
  h->cfg = *cfg;
  h->device = device;
  DevParams& p = h->p;
  const int B = cfg->num_envs, N = cfg->num_agents, O = cfg->num_obstacles, W = cfg->num_walls, E = 2 * N + O + W;
  p.B = B; p.N = N; p.O = O; p.E = E; p.W = W;
  p.env_begin = 0; p.env_end = B;
  p.Bp = (B + 63) & ~63;
  const size_t Bp = (size_t)p.Bp;
  const int SP = (N + O + W) * (N + O + W - 1) / 2;    // static entities: landmarks, obstacles, walls
  const int SPp = (SP + 3) & ~3;                   // per-env row of the group mapping's layout
  const size_t words = Bp * (size_t)(9 * N + 3 * N + 2 * N + 2 * O + 4 + SPp + 2 * W + 1);
  cudaError_t e = cudaMalloc(&h->state_block, words * 4);
  if (e != cudaSuccess) { delete h; return fail(FM_ERR_CUDA, "fm_create: cudaMalloc(%zu B): %s", words * 4, cudaGetErrorString(e)); }
  cudaMemset(h->state_block, 0, words * 4);
  float* f = (float*)h->state_block;
  auto take = [&](size_t n) { float* r = f; f += n; return r; };
  p.px = take(Bp * N); p.py = take(Bp * N); p.vx = take(Bp * N); p.vy = take(Bp * N); p.pdist = take(Bp * N);
  p.dtg = take(Bp * N); p.treq = take(Bp * N); p.dleft = take(Bp * N); p.mintime = take(Bp * N);
  p.gm = (int*)take(Bp * N); p.nac = (int*)take(Bp * N); p.noc = (int*)take(Bp * N);
  p.lx = take(Bp * N); p.ly = take(Bp * N);
  p.ox = take(Bp * O); p.oy = take(Bp * O);
  p.dmean = take(Bp); p.dstd = take(Bp); p.step = (int*)take(Bp); p.episode = (int*)take(Bp);
  p.sdist = take(Bp * SPp);
  p.wax = take(Bp * W); p.wor = (int*)take(Bp * W); p.wlen = take(Bp);     // after sdist: the agent-warp kernels index rows up to sdist

  // config -> device constants.  Collision threshold exactly as the reference spells it:
  // 1.05*(size + size) (navigation_graph.py:655, :704); cached min_dist = size + size (core.py:215).
  const double size = 0.05;
  p.min_dist_thresh = cfg->min_dist_thresh;
  p.dcoll = 1.05 * (size + size);
  p.max_speed = cfg->max_speed;
  p.has_max_speed = cfg->max_speed > 0.0;
  p.dt = 0.1;
  p.damping_keep = 1 - 0.25;
  p.zeroshift = cfg->zeroshift;
  p.zeroshift_f = (float)cfg->zeroshift;
  p.fair_rew_d = cfg->fair_rew;
  p.goal_rew = (float)cfg->goal_rew;
  p.coll_rew = (float)cfg->collision_rew;
  p.fair_rew = (float)cfg->fair_rew;
  p.world_size = (float)cfg->world_size;
  p.half_world = (float)(cfg->world_size / 2);
  p.clip_lo = (float)(-2 * cfg->collision_rew);             // navigation_graph.py:824
  p.clip_hi = (float)(cfg->goal_rew + cfg->fair_rew);
  p.contact_force = 3e2f;                                    // core.py:153-160
  p.contact_margin = 2e-2f;
  p.dist_min = (float)(size + size);
  p.inv_margin = 1.0f / p.contact_margin;
  p.cf_margin = p.contact_force * p.contact_margin;
  {                                                          // largest double whose sqrt is <= max_speed
    double t = cfg->max_speed * cfg->max_speed;
    if (p.has_max_speed) {
      while (sqrt(t) > cfg->max_speed) t = nextafter(t, 0.0);
      while (sqrt(nextafter(t, INFINITY)) <= cfg->max_speed) t = nextafter(t, INFINITY);
    }
    p.speed2_max = t;
  }
  {                                                          // smallest double whose sqrt is >= dcoll: sqrt_rn(x) < dcoll  <=>  x < dcoll2_lt
    double t = p.dcoll * p.dcoll;
    while (sqrt(t) < p.dcoll) t = nextafter(t, INFINITY);
    while (sqrt(nextafter(t, 0.0)) >= p.dcoll) t = nextafter(t, 0.0);
    p.dcoll2_lt = t;
  }
  p.episode_length = cfg->episode_length;
  p.fairness_reward = cfg->fairness_reward;
  p.collaborative = cfg->collaborative;
  p.auto_reset = cfg->auto_reset;
  p.info_every_step = cfg->info_every_step;
  p.feat_global = cfg->graph_feat_global ? 1 : 0;
  p.seed_lo = (uint32_t)(cfg->seed & 0xffffffffull);
  p.seed_hi = (uint32_t)(cfg->seed >> 32);
  p.env_offset = cfg->env_offset;

  // Kernel mapping (cfg->mapping: 0 auto = agent-warp where compiled for (N, O), else group-per-env;
  // 1 group-per-env; 2 agent-warp).  Both mappings produce identical results.
  if (cfg->mapping == 2 && !fm::aw_supported(N, O, W)) {
    cudaFree(h->state_block); delete h;
    return fail(FM_ERR_UNSUPPORTED, "fm_create: agent-warp kernels are not compiled for N=%d O=%d", N, O);
  }
  p.mapping = cfg->mapping == 1 ? 0 : ((cfg->mapping == 2 || fm::aw_supported(N, O, W)) ? 1 : 0);
  p.sd_env_stride = p.mapping == 0 ? SPp : 0;      // group mapping: [env][SPp];  agent-warp mapping: [pair][Bp]
  // pending block of the next-episode prefetch (group mapping with auto-reset; FM_PREFETCH=0 disables it)
  h->lockstep = 1; h->host_step = 0;
  {
    const char* ev = getenv("FM_PREFETCH");
    // Group mapping: on unless FM_PREFETCH=0.  Agent-warp mapping: the kernels consume the same block (bit-identical,
    // tested), but only with FM_PREFETCH=2: measured SLOWER at C2 (0.767 vs 0.861 of the roofline in the driver
    // configuration, 0.80 vs 0.93 in long runs, profiles/r02_u_*).  There the inline reset costs 47 us per episode with
    // lane = env (32 envs per warp in lockstep), while prefetch_kernel<4> spends 4 lanes per env on the same serial work and
    // takes the SMs from the memory-bound step kernels it runs beside.
    const int v = ev ? atoi(ev) : 1;
    h->pf_on = cfg->auto_reset && (p.mapping == 0 ? v != 0 : (v == 2 && W == 0));   // (the agent-warp wall kernels reset inline)
  }
  if (h->pf_on) {
    const size_t rows = (size_t)(5 * N + 2 * O + 2 * W);
    e = cudaMalloc(&h->pend_block, (rows * Bp + Bp) * 4);
    if (e != cudaSuccess) { cudaFree(h->state_block); delete h; return fail(FM_ERR_CUDA, "fm_create: cudaMalloc pending block: %s", cudaGetErrorString(e)); }
    float* g = (float*)h->pend_block;
    auto takeq = [&](size_t n) { float* r = g; g += n; return r; };
    p.q_px = takeq(Bp * N); p.q_py = takeq(Bp * N); p.q_lx = takeq(Bp * N); p.q_ly = takeq(Bp * N);
    p.q_ox = takeq(Bp * O); p.q_oy = takeq(Bp * O); p.q_gm = (int*)takeq(Bp * N);
    p.q_wax = takeq(Bp * W); p.q_wor = (int*)takeq(Bp * W); p.q_tag = (int*)takeq(Bp);
    cudaMemset(p.q_tag, 0xff, Bp * 4);              // -1: no entry
  }
  const int G = fm::group_size(N), EPW = 32 / G;
  p.sm_cost = 0;                                   // the reset's cost matrix lives inside the adj tile
  p.sm_ent = round4((long long)EPW * E * fm::ENT_STRIDE);
  // adj / obs images sit at the 16-byte phase of their destinations (<= 3 words of slack); the adj region is
  // reused as two node_obs staging buffers of stage_k x 32 rows (+ phase slack) each, so it holds at least 2 x 1.
  const int stage_words = fm::STAGE_SUB * fm::NODE_F;                  // 352
  // node_obs staging inside the adj region: two buffers of 96 rows if they fit, else ONE buffer of 96 rows (refilled
  // once the copy engine has read it: fewer, larger chunks beat double buffering when the region is small -- N = 7),
  // else two buffers of 32 rows.  FM_STAGE=k3x2|k3x1|k1x2 forces a variant (diagnostic; may enlarge the region).
  const char* force = getenv("FM_STAGE");
  long long need = (long long)EPW * E * E + 3;
  if (force && !strcmp(force, "k3x2")) need = std::max(need, 2LL * (3 * stage_words + 4));
  p.sm_adj = round4(std::max(need, 2LL * (stage_words + 4)));
  const int half = (p.sm_adj >> 1) & ~3;
  if (half - 3 >= 3 * stage_words) { p.stage_k = 3; p.stage_bufs = 2; }
  else if (p.sm_adj - 3 >= 3 * stage_words) { p.stage_k = 3; p.stage_bufs = 1; }
  else { p.stage_k = 1; p.stage_bufs = 2; }
  if (force && !strcmp(force, "k1x2")) { p.stage_k = 1; p.stage_bufs = 2; }
  if (force && !strcmp(force, "k3x1") && p.sm_adj - 3 >= 3 * stage_words) { p.stage_k = 3; p.stage_bufs = 1; }
  p.sm_obs = round4((long long)EPW * N * fm::OBS_F + 3);
  p.sm_asg = round4((long long)EPW * N);               // lexifair row masks (the matching lives in registers)
  p.sm_per_warp = p.sm_cost + p.sm_ent + p.sm_adj + p.sm_obs + p.sm_asg;
  p.sm_pf_cost = round4(2LL * N * N + (N * N + 1) / 2 + 2);          // float64 costs | uint16 permutation | alignment
  p.sm_pf_per_warp = EPW * p.sm_pf_cost + p.sm_ent + p.sm_asg;
  if (p.mapping == 0 && (size_t)p.sm_per_warp * 4 * 4 > 227 * 1024) {
    cudaFree(h->pend_block); cudaFree(h->state_block); delete h;
    return fail(FM_ERR_UNSUPPORTED, "fm_create: N=%d O=%d needs %d B of shared memory per CTA", N, O, p.sm_per_warp * 16);
  }
  h->K = fm_stats_len(N);
  h->stats_rows = p.mapping == 1 ? fm::aw_stats_rows(B) : fm::num_warps(B, N);
  e = cudaMalloc(&h->stats, (size_t)h->stats_rows * h->K * sizeof(double));
  if (e != cudaSuccess) { cudaFree(h->state_block); delete h; return fail(FM_ERR_CUDA, "fm_create: cudaMalloc stats: %s", cudaGetErrorString(e)); }
  cudaMemset(h->stats, 0, (size_t)h->stats_rows * h->K * sizeof(double));
  p.stats = h->stats;
  e = fm::prepare_kernels(p);
  if (e != cudaSuccess) { cudaFree(h->stats); cudaFree(h->pend_block); cudaFree(h->state_block); delete h; return fail(FM_ERR_CUDA, "fm_create: kernel attributes: %s", cudaGetErrorString(e)); }
  if (const char* ev = getenv("FM_LANES")) {          // diagnostic override of the env-range lanes of fm_step_many
    const int v = atoi(ev);
    if (v >= 1 && v <= FM_MAX_LANES) h->lanes_override = v;
  }
  if (p.mapping == 1) {
    // Persistent rollout kernel (fm_roll.cu), opt-in with FM_ROLL=1.  Measured on B200 at C2 it reaches 70 % of the HBM
    // roofline against 93 % for the one-shot kernels on two env-range lanes replayed from a CUDA graph (profiles/r02_*), so
    // the one-shot kernels stay the default path; the rollout kernel is kept, tested, for single-launch use.
    const char* ev = getenv("FM_ROLL");
    h->roll_on = ev && atoi(ev) != 0 && W == 0;      // (no wall instantiation of the rollout kernel)
    int per_sm = 0, sms = 0;
    e = fm::roll_prepare(p, &per_sm);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaMalloc(&h->roll_ctl, fm::roll_ctl_bytes(B));
    if (e == cudaSuccess) e = cudaMemset(h->roll_ctl, 0, fm::roll_ctl_bytes(B));
    if (e != cudaSuccess || per_sm < 1) {
      cudaFree(h->roll_ctl); cudaFree(h->stats); cudaFree(h->pend_block); cudaFree(h->state_block); delete h;
      return fail(FM_ERR_CUDA, "fm_create: rollout kernel: %s", cudaGetErrorString(e));
    }
    h->roll_max_ctas = per_sm * sms;
    if (const char* ev2 = getenv("FM_ROLL_CTAS")) { const int v = atoi(ev2); if (v >= 1) h->roll_max_ctas = v; }   // diagnostic
    // start-up stagger of the CTAs of an SM (fm_roll.cu), only when the launch has several items per CTA
    h->roll_stagger_ns = 0; h->roll_stagger1_ns = 0;
    if (const char* ev3 = getenv("FM_ROLL_STAGGER_NS")) h->roll_stagger_ns = atoi(ev3);
    if (const char* ev4 = getenv("FM_ROLL_STAGGER1_NS")) h->roll_stagger1_ns = atoi(ev4);
  }
  e = fm::launch_state_init(p, 0);
  if (e == cudaSuccess) e = cudaStreamSynchronize(0);
  if (e != cudaSuccess) { cudaFree(h->stats); cudaFree(h->pend_block); cudaFree(h->state_block); delete h; return fail(FM_ERR_CUDA, "fm_create: init: %s", cudaGetErrorString(e)); }
  h->launches = 1;
  *out = h;
  return FM_OK;
}

static void free_staging(FmHandle* h) {
  if (!h->staging) return;
  cudaFree(h->st_onehot); cudaFree(h->st_mask);
  cudaFree(h->st_out.obs); cudaFree(h->st_out.node_obs); cudaFree(h->st_out.adj);
  cudaFree(h->st_out.reward); cudaFree(h->st_out.done); cudaFree(h->st_out.info);
  h->staging = false;
}

int fm_destroy(FmHandle* h) {
  if (!h) return FM_OK;
  use_device(h->device);
  free_staging(h);
  if (h->pf_ready_made) {
    for (int k = 0; k < FM_MAX_LANES; ++k) { cudaStreamDestroy(h->pf_stream[k]); cudaEventDestroy(h->pf_go[k]); cudaEventDestroy(h->pf_ready[k]); }
  }
  cudaFree(h->pend_block);
  if (h->lanes_ready) {
    for (int k = 1; k < FM_MAX_LANES; ++k) { cudaStreamDestroy(h->lane_stream[k]); cudaEventDestroy(h->lane_join[k]); }
    cudaEventDestroy(h->lane_fork);
  }
  cudaFree(h->roll_ctl);
  cudaFree(h->stats);
  cudaFree(h->state_block);
  delete h;
  return FM_OK;
}

static void set_outputs(DevParams& p, const FmOutputs* out) {
  p.o_obs = out ? out->obs : nullptr;
  p.o_node = out ? out->node_obs : nullptr;
  p.o_adj = out ? out->adj : nullptr;
  p.o_rew = out ? out->reward : nullptr;
  p.o_done = out ? out->done : nullptr;
  p.o_info = out ? out->info : nullptr;
}

// ---- next-episode prefetch plumbing -----------------------------------------------------------------------------
static bool stream_capturing(cudaStream_t s) {
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(s, &st) != cudaSuccess) { cudaGetLastError(); return false; }
  return st != cudaStreamCaptureStatusNone;
}

static int ensure_prefetch_streams(FmHandle* h) {
  if (h->pf_ready_made) return FM_OK;
  // Most urgent priority: the prefetch is a fixed amount of SM work that has to be done before the next terminal
  // step either way; running it first (at 7+ CTAs/SM) measured slightly better than letting it trail behind the
  // step kernels (C3 66 % vs 64 % of the roofline), and the terminal step never waits.  FM_PREFETCH_PRIO=0: least urgent.
  int lo = 0, hi = 0;
  FM_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));       // lo = least urgent, hi = most urgent
  int prio = hi;
  if (const char* ev = getenv("FM_PREFETCH_PRIO")) { if (atoi(ev) == 0) prio = lo; }
  for (int k = 0; k < FM_MAX_LANES; ++k) {
    FM_CUDA(cudaStreamCreateWithPriority(&h->pf_stream[k], cudaStreamNonBlocking, prio));
    FM_CUDA(cudaEventCreateWithFlags(&h->pf_go[k], cudaEventDisableTiming));
    FM_CUDA(cudaEventCreateWithFlags(&h->pf_ready[k], cudaEventDisableTiming));
  }
  h->pf_ready_made = 1;
  return FM_OK;
}

// Before a step launch on stream s: the kernel may consume pending entries only when the host knows the episode
// phase (lockstep) and the stream is not being captured; a terminal step waits for every prefetch in flight.
static int prefetch_before_step(FmHandle* h, DevParams& p, cudaStream_t s, bool terminal) {
  // The kernels take an entry only if its tag equals the env's episode key (acquire load), and an entry depends on (seed,
  // global env, key) alone: consuming it needs no host knowledge.  What the host's view of the phase (lockstep, not
  // capturing) adds is the wait that makes sure the prefetch launched after the last terminal step has finished.
  if (!h->pf_on) { p.q_tag = nullptr; return FM_OK; }
  if (!h->lockstep || stream_capturing(s)) return FM_OK;
  if (terminal)
    for (int k = 0; k < FM_MAX_LANES; ++k)
      if (h->pf_used[k]) FM_CUDA(cudaStreamWaitEvent(s, h->pf_ready[k], 0));
  return FM_OK;
}

// After a launch on stream s that advanced the episode counters of envs [env_begin, env_end): produce their next
// placement + assignment on lane `lane`'s low-priority side stream.
static int prefetch_after_reset(FmHandle* h, cudaStream_t s, int lane, int env_begin, int env_end) {
  if (!h->pf_on || !h->lockstep || stream_capturing(s)) return FM_OK;
  int rc = ensure_prefetch_streams(h);
  if (rc) return rc;
  FM_CUDA(cudaEventRecord(h->pf_go[lane], s));
  FM_CUDA(cudaStreamWaitEvent(h->pf_stream[lane], h->pf_go[lane], 0));
  DevParams p = h->p;
  p.env_begin = env_begin; p.env_end = env_end;
  FM_CUDA(fm::launch_prefetch(p, h->pf_stream[lane]));
  FM_CUDA(cudaEventRecord(h->pf_ready[lane], h->pf_stream[lane]));
  h->pf_used[lane] = 1;
  h->launches += 1;
  return FM_OK;
}

// Host view of the episode phase: returns whether the step about to be launched is terminal for every env.
static bool step_is_terminal(const FmHandle* h) { return h->lockstep && h->host_step + 1 >= h->p.episode_length; }
static void advance_phase(FmHandle* h, bool terminal) {
  if (!h->lockstep) return;
  if (!terminal) { h->host_step += 1; return; }
  if (h->p.auto_reset) h->host_step = 0; else h->lockstep = 0;
}

int fm_observe(FmHandle* h, const FmOutputs* out, void* stream) {
  if (!h) return fail(FM_ERR_INVALID_ARG, "fm_observe: null handle");
  int rc = use_device(h->device);
  if (rc) return rc;
  DevParams p = h->p;
  set_outputs(p, out);
  p.reset_mask = nullptr; p.observe_only = 1;
  p.act_idx = nullptr; p.act_onehot = nullptr;
  FM_CUDA(fm::launch_step(p, (cudaStream_t)stream, true));
  h->launches += 1;
  return FM_OK;                                      // no state change: the episode phase the host tracks stays valid
}

int fm_soa_stride(const FmHandle* h) { return h ? h->p.Bp : 0; }

int fm_observe_soa(FmHandle* h, const FmSoaOutputs* out, void* stream) {
  if (!h || !out) return fail(FM_ERR_INVALID_ARG, "fm_observe_soa: null argument");
  if (h->p.W > 0) return fail(FM_ERR_UNSUPPORTED, "fm_observe_soa: walls are not supported in the SoA mode");
  for (const float* q : {out->obs, out->node_obs, out->adj})
    if (q && (reinterpret_cast<uintptr_t>(q) & 15u)) return fail(FM_ERR_INVALID_ARG, "fm_observe_soa: outputs must be 16-byte aligned");
  int rc = use_device(h->device);
  if (rc) return rc;
  FM_CUDA(fm::launch_observe_soa(h->p, out->obs, out->node_obs, out->adj, (cudaStream_t)stream));
  h->launches += 1;
  return FM_OK;
}

int fm_check_finite(FmHandle* h, int32_t* flags, int32_t* count, void* stream) {
  if (!h) return fail(FM_ERR_INVALID_ARG, "fm_check_finite: null handle");
  int rc = use_device(h->device);
  if (rc) return rc;
  FM_CUDA(fm::launch_finite_guard(h->p, flags, count, (cudaStream_t)stream));
  h->launches += 1;
  return FM_OK;
}

int fm_reset(FmHandle* h, const uint8_t* mask, const FmOutputs* out, void* stream) {
  if (!h) return fail(FM_ERR_INVALID_ARG, "fm_reset: null handle");
  int rc = use_device(h->device);
  if (rc) return rc;
  DevParams p = h->p;
  set_outputs(p, out);
  p.reset_mask = mask;
  p.act_idx = nullptr; p.act_onehot = nullptr;
  FM_CUDA(fm::launch_step(p, (cudaStream_t)stream, true));
  h->launches += 1;
  if (mask) h->lockstep = 0;                         // envs are no longer in the same episode phase
  else { h->lockstep = 1; h->host_step = 0; }
  return prefetch_after_reset(h, (cudaStream_t)stream, 0, 0, h->p.B);
}

// Side streams + fork / join events shared by fm_step_many (env-range lanes) and the host-buffer copies.
static int ensure_lanes(FmHandle* h) {
  if (h->lanes_ready) return FM_OK;
  h->lane_stream[0] = nullptr;
  for (int k = 1; k < FM_MAX_LANES; ++k) {
    FM_CUDA(cudaStreamCreateWithFlags(&h->lane_stream[k], cudaStreamNonBlocking));
    FM_CUDA(cudaEventCreateWithFlags(&h->lane_join[k], cudaEventDisableTiming));
  }
  FM_CUDA(cudaEventCreateWithFlags(&h->lane_fork, cudaEventDisableTiming));
  h->lanes_ready = 1;
  return FM_OK;
}

static int step_common(FmHandle* h, const int32_t* idx, const float* onehot, const FmOutputs* out, void* stream) {
  if (!h) return fail(FM_ERR_INVALID_ARG, "fm_step: null handle");
  if (!idx && !onehot) return fail(FM_ERR_INVALID_ARG, "fm_step: null actions");
  int rc = use_device(h->device);
  if (rc) return rc;
  DevParams p = h->p;
  set_outputs(p, out);
  p.act_idx = idx; p.act_onehot = onehot; p.reset_mask = nullptr;
  // A captured launch is replayed without passing through here: the host's view of the episode phase would drift, so
  // the next-episode prefetch (the only consumer of that view) stays off until the next full fm_reset.
  if (stream_capturing((cudaStream_t)stream)) h->lockstep = 0;
  const bool terminal = step_is_terminal(h);
  rc = prefetch_before_step(h, p, (cudaStream_t)stream, terminal);
  if (rc) return rc;
  if (h->roll_on) {                                  // agent-warp mapping: one-step launch of the persistent kernel
    FmOutputs o{p.o_obs, p.o_node, p.o_adj, p.o_rew, p.o_done, p.o_info};
    const int tiles = (h->p.B + 31) / 32;
    fm::RollLaunch r{1, 1, h->roll_max_ctas, tiles > h->roll_max_ctas ? h->roll_stagger1_ns : 0, h->roll_ctl, idx, onehot, 0, &o};
    FM_CUDA(fm::roll_launch(p, r, (cudaStream_t)stream));
  } else {
    // one launch per step (the closed loop): let the next step's kernel be scheduled behind this one's last wave
    // (programmatic dependent launch; 26.7 -> 25.3 us per step at C2, profiles/r02_pdl_*; FM_STEP_PDL=0: plain stream order)
    static const int step_pdl = [] { const char* v = getenv("FM_STEP_PDL"); return (v && v[0] == '0') ? 0 : 1; }();
    p.pdl = step_pdl && p.mapping == 1 && !stream_capturing((cudaStream_t)stream);
    FM_CUDA(fm::launch_step(p, (cudaStream_t)stream, false));
  }
  h->launches += 1;
  advance_phase(h, terminal);
  if (terminal && h->p.auto_reset) return prefetch_after_reset(h, (cudaStream_t)stream, 0, 0, h->p.B);
  return FM_OK;
}

int fm_step(FmHandle* h, const int32_t* actions, const FmOutputs* out, void* stream) {
  return step_common(h, actions, nullptr, out, stream);
}

int fm_step_onehot(FmHandle* h, const float* onehot, const FmOutputs* out, void* stream) {
  return step_common(h, nullptr, onehot, out, stream);
}

int fm_step_many(FmHandle* h, const int32_t* actions, int32_t num_steps, const FmOutputs* outs, void* stream) {
  if (!h || !actions || !outs) return fail(FM_ERR_INVALID_ARG, "fm_step_many: null argument");
  if (num_steps < 0) return fail(FM_ERR_INVALID_ARG, "fm_step_many: num_steps < 0");
  int rc = use_device(h->device);
  if (rc) return rc;
  const size_t stride = (size_t)h->p.B * h->p.N;
  const bool capturing = stream_capturing((cudaStream_t)stream);
  if (capturing) h->lockstep = 0;                                   // see step_common
  if (h->roll_on) {
    // Agent-warp mapping: the whole rollout is (step, tile) items of ONE persistent kernel per chunk of <=
    // FM_ROLL_MAX_STEPS steps (fm_roll.cu).  A tile's next step may start as soon as its state is written back when
    // every step of the chunk has its own output arrays; otherwise only after its outputs have been written.
    for (int t0 = 0; t0 < num_steps; t0 += FM_ROLL_MAX_STEPS) {
      const int n = std::min(FM_ROLL_MAX_STEPS, num_steps - t0);
      int early = 1;
      for (int a = 0; a < n && early; ++a)
        for (int b = a + 1; b < n && early; ++b) {
          const FmOutputs &x = outs[t0 + a], &y = outs[t0 + b];
          if ((x.obs && x.obs == y.obs) || (x.node_obs && x.node_obs == y.node_obs) || (x.adj && x.adj == y.adj) ||
              (x.reward && x.reward == y.reward) || (x.done && x.done == y.done)) early = 0;
        }
      DevParams p = h->p;
      set_outputs(p, nullptr);
      p.act_idx = nullptr; p.act_onehot = nullptr; p.reset_mask = nullptr;
      const long long items = (long long)n * ((h->p.B + 31) / 32);
      fm::RollLaunch r{n, early, h->roll_max_ctas, items > 2LL * h->roll_max_ctas ? h->roll_stagger_ns : 0, h->roll_ctl,
                       actions + (size_t)t0 * stride, nullptr, (long long)stride, outs + t0};
      FM_CUDA(fm::roll_launch(p, r, (cudaStream_t)stream));
      h->launches += 1;
      for (int t = 0; t < n; ++t) advance_phase(h, step_is_terminal(h));
    }
    return FM_OK;
  }
  // Envs are independent, so a rollout of T steps is T x L independent kernel chains, one per env-range
  // lane.  Lane 0 runs on the caller's stream, the others on side streams forked from / joined to it; the
  // GPU then always has runnable CTAs of another lane while one lane's last wave drains or its next
  // launch is in flight.  Small batches (less than two waves of CTAs per lane) stay on one stream.
  const int B = h->p.B;
  int lanes = 1;
  if (num_steps > 1 && B >= 32768) lanes = 2;           // 2, 3, 4 lanes measure the same at C2; 8 is launch bound
  if (h->lanes_override) lanes = h->lanes_override;                   // FM_LANES, diagnostic
  if (lanes > 1) { rc = ensure_lanes(h); if (rc) return rc; }
  cudaStream_t user = (cudaStream_t)stream;
  if (lanes > 1) {
    FM_CUDA(cudaEventRecord(h->lane_fork, user));
    for (int k = 1; k < lanes; ++k) FM_CUDA(cudaStreamWaitEvent(h->lane_stream[k], h->lane_fork, 0));
  }
  const int per_lane = (((B + lanes - 1) / lanes) + 127) & ~127;      // lane boundaries at multiples of 128 envs
  // Next-episode prefetch when the host does not drive it (stream capture, or the episode phase unknown to the host): one
  // launch per lane at the START of the call, on the lane's prefetch stream, joined at the end of the call (so that a
  // capture closes).  It redraws the entries whose tag is stale -- all of them right after a terminal step, none
  // otherwise -- so a rollout issued in calls that start behind episode boundaries (bench.py, the rollout buffer) finds
  // the entries at its terminal steps; any other call pattern falls back to the inline reset, entry by entry.
  const bool pf_call = h->pf_on && num_steps > 0 && (!h->lockstep || stream_capturing(user));
  if (pf_call) {
    rc = ensure_prefetch_streams(h);
    if (rc) return rc;
    for (int k = 0; k < lanes; ++k) {
      DevParams p = h->p;
      p.env_begin = k * per_lane < B ? k * per_lane : B;
      p.env_end = (k + 1) * per_lane < B ? (k + 1) * per_lane : B;
      if (p.env_begin >= p.env_end) continue;
      cudaStream_t ls = k == 0 ? user : h->lane_stream[k];
      FM_CUDA(cudaEventRecord(h->pf_go[k], ls));
      FM_CUDA(cudaStreamWaitEvent(h->pf_stream[k], h->pf_go[k], 0));
      FM_CUDA(fm::launch_prefetch(p, h->pf_stream[k]));
      FM_CUDA(cudaEventRecord(h->pf_ready[k], h->pf_stream[k]));
      h->launches += 1;
    }
  }
  for (int t = 0; t < num_steps; ++t) {
    const bool terminal = step_is_terminal(h);
    for (int k = 0; k < lanes; ++k) {
      DevParams p = h->p;
      set_outputs(p, outs + t);
      p.act_idx = actions + (size_t)t * stride; p.act_onehot = nullptr; p.reset_mask = nullptr;
      p.env_begin = k * per_lane < B ? k * per_lane : B;
      p.env_end = (k + 1) * per_lane < B ? (k + 1) * per_lane : B;
      if (p.env_begin >= p.env_end) continue;
      cudaStream_t ls = k == 0 ? user : h->lane_stream[k];
      rc = prefetch_before_step(h, p, ls, terminal);
      if (rc) return rc;
      // The lane's consecutive step kernels as programmatic dependent launches when they are issued eagerly: long run 0.954 ->
      // 0.975 of the roofline on the same box.  Not under capture (FM_MANY_PDL=2 forces it there: the replayed driver
      // configuration measured 0.851 / 0.880 with the programmatic edges against 0.855 / 0.890 without, profiles/r02_pdl2_*).
      static const int many_pdl = [] { const char* v = getenv("FM_MANY_PDL"); return v && v[0] ? atoi(v) : 1; }();
      p.pdl = p.mapping == 1 && (many_pdl == 2 || (many_pdl == 1 && !capturing));
      FM_CUDA(fm::launch_step(p, ls, false));
      h->launches += 1;
      if (terminal && h->p.auto_reset) { rc = prefetch_after_reset(h, ls, k, p.env_begin, p.env_end); if (rc) return rc; }
    }
    advance_phase(h, terminal);
  }
  if (pf_call)
    for (int k = 0; k < lanes; ++k)
      if ((k * per_lane < B ? k * per_lane : B) < ((k + 1) * per_lane < B ? (k + 1) * per_lane : B))
        FM_CUDA(cudaStreamWaitEvent(k == 0 ? user : h->lane_stream[k], h->pf_ready[k], 0));
  if (lanes > 1) {
    for (int k = 1; k < lanes; ++k) {
      FM_CUDA(cudaEventRecord(h->lane_join[k], h->lane_stream[k]));
      FM_CUDA(cudaStreamWaitEvent(user, h->lane_join[k], 0));
    }
  }
  return FM_OK;
}

static int ensure_staging(FmHandle* h) {
  if (h->staging) return FM_OK;
  const size_t B = h->p.B, N = h->p.N, E = h->p.E;
  FM_CUDA(cudaMalloc(&h->st_onehot, B * N * 5 * sizeof(float)));
  FM_CUDA(cudaMalloc(&h->st_mask, B));
  FM_CUDA(cudaMalloc(&h->st_out.obs, B * N * fm::OBS_F * sizeof(float)));
  FM_CUDA(cudaMalloc(&h->st_out.node_obs, B * N * E * fm::NODE_F * sizeof(float)));
  FM_CUDA(cudaMalloc(&h->st_out.adj, B * E * E * sizeof(float)));
  FM_CUDA(cudaMalloc(&h->st_out.reward, B * N * sizeof(float)));
  FM_CUDA(cudaMalloc(&h->st_out.done, B * N));
  FM_CUDA(cudaMalloc(&h->st_out.info, B * N * fm::INFO_F * sizeof(float)));
  FM_CUDA(cudaMemset(h->st_out.info, 0, B * N * fm::INFO_F * sizeof(float)));
  h->staging = true;
  return FM_OK;
}

// Device staging -> caller's host buffers.  One D2H stream reaches ~52 GB/s on this PCIe link, two concurrent ones
// ~55 GB/s (two copy engines), so large results are split over the caller's stream and one side stream (about half
// of the bytes each: the side stream takes adj and the tail of node_obs) and joined before returning.
static int copy_outputs_to_host(FmHandle* h, const FmOutputs* out_host, bool with_step_outputs, cudaStream_t st) {
  const size_t B = h->p.B, N = h->p.N, E = h->p.E;
  if (!out_host) return FM_OK;
  const size_t node_bytes = B * N * E * (h->p.feat_global ? fm::NODE_F_GLOBAL : fm::NODE_F) * 4, adj_bytes = B * E * E * 4;
  const size_t small_bytes = B * N * (fm::OBS_F * 4 + 5);
  size_t node_side = 0;                              // bytes of node_obs copied by the side stream
  cudaStream_t side = st;
  const bool split = out_host->node_obs && node_bytes + adj_bytes > (8u << 20);
  if (split) {
    int rc = ensure_lanes(h);
    if (rc) return rc;
    side = h->lane_stream[1];
    const size_t total = node_bytes + (out_host->adj ? adj_bytes : 0) + small_bytes;
    const size_t side_adj = out_host->adj ? adj_bytes : 0;
    node_side = total / 2 > side_adj ? ((total / 2 - side_adj) & ~(size_t)15) : 0;
    if (node_side > node_bytes) node_side = node_bytes;
    FM_CUDA(cudaEventRecord(h->lane_fork, st));
    FM_CUDA(cudaStreamWaitEvent(side, h->lane_fork, 0));
  }
  if (out_host->node_obs) {
    FM_CUDA(cudaMemcpyAsync(out_host->node_obs, h->st_out.node_obs, node_bytes - node_side, cudaMemcpyDeviceToHost, st));
    if (node_side)
      FM_CUDA(cudaMemcpyAsync((char*)out_host->node_obs + (node_bytes - node_side), (char*)h->st_out.node_obs + (node_bytes - node_side),
                              node_side, cudaMemcpyDeviceToHost, side));
  }
  if (out_host->adj) FM_CUDA(cudaMemcpyAsync(out_host->adj, h->st_out.adj, adj_bytes, cudaMemcpyDeviceToHost, side));
  if (out_host->obs) FM_CUDA(cudaMemcpyAsync(out_host->obs, h->st_out.obs, B * N * fm::OBS_F * 4, cudaMemcpyDeviceToHost, st));
  if (with_step_outputs) {
    if (out_host->reward) FM_CUDA(cudaMemcpyAsync(out_host->reward, h->st_out.reward, B * N * 4, cudaMemcpyDeviceToHost, st));
    if (out_host->done) FM_CUDA(cudaMemcpyAsync(out_host->done, h->st_out.done, B * N, cudaMemcpyDeviceToHost, st));
    if (out_host->info) FM_CUDA(cudaMemcpyAsync(out_host->info, h->st_out.info, B * N * fm::INFO_F * 4, cudaMemcpyDeviceToHost, st));
  }
  if (split) {
    FM_CUDA(cudaEventRecord(h->lane_join[1], side));
    FM_CUDA(cudaStreamWaitEvent(st, h->lane_join[1], 0));
  }
  return FM_OK;
}

int fm_step_host(FmHandle* h, const float* onehot_host, const FmOutputs* out_host, void* stream) {
  if (!h || !onehot_host) return fail(FM_ERR_INVALID_ARG, "fm_step_host: null argument");
  int rc = use_device(h->device);
  if (rc) return rc;
  rc = ensure_staging(h);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t B = h->p.B, N = h->p.N;
  FM_CUDA(cudaMemcpyAsync(h->st_onehot, onehot_host, B * N * 5 * sizeof(float), cudaMemcpyHostToDevice, st));
  FmOutputs dev = h->st_out;
  rc = step_common(h, nullptr, h->st_onehot, &dev, stream);
  if (rc) return rc;
  rc = copy_outputs_to_host(h, out_host, true, st);
  if (rc) return rc;
  FM_CUDA(cudaStreamSynchronize(st));
  return FM_OK;
}

static void host_lane_range(const FmHandle* h, int lane, int num_lanes, int& b0, int& b1) {
  const int B = h->p.B;
  const int per = (((B + num_lanes - 1) / num_lanes) + 127) & ~127;
  b0 = lane * per < B ? lane * per : B;
  b1 = (lane + 1) * per < B ? (lane + 1) * per : B;
}

int fm_host_lane_range(const FmHandle* h, int32_t lane, int32_t num_lanes, int32_t* env_begin, int32_t* env_end) {
  if (!h || !env_begin || !env_end || num_lanes < 1 || num_lanes > FM_MAX_LANES || lane < 0 || lane >= num_lanes)
    return fail(FM_ERR_INVALID_ARG, "fm_host_lane_range: bad arguments");
  int b0, b1;
  host_lane_range(h, lane, num_lanes, b0, b1);
  *env_begin = b0; *env_end = b1;
  return FM_OK;
}

int fm_step_host_lane(FmHandle* h, const float* onehot_host, const FmOutputs* out_host, int32_t lane, int32_t num_lanes, void* stream) {
  if (!h || !onehot_host) return fail(FM_ERR_INVALID_ARG, "fm_step_host_lane: null argument");
  if (num_lanes < 1 || num_lanes > FM_MAX_LANES || lane < 0 || lane >= num_lanes) return fail(FM_ERR_INVALID_ARG, "fm_step_host_lane: bad lane");
  if (h->roll_on) return fail(FM_ERR_UNSUPPORTED, "fm_step_host_lane: not available with FM_ROLL=1");
  int rc = use_device(h->device);
  if (rc) return rc;
  rc = ensure_staging(h);
  if (rc) return rc;
  rc = ensure_lanes(h);
  if (rc) return rc;
  cudaStream_t user = (cudaStream_t)stream;
  cudaStream_t ls = lane == 0 ? user : h->lane_stream[lane];
  if (lane == 0 && num_lanes > 1) FM_CUDA(cudaEventRecord(h->lane_fork, user));
  if (lane > 0) FM_CUDA(cudaStreamWaitEvent(ls, h->lane_fork, 0));
  int b0, b1;
  host_lane_range(h, lane, num_lanes, b0, b1);
  const bool terminal = step_is_terminal(h);
  if (b0 < b1) {
    const size_t N = h->p.N, E = h->p.E, n = (size_t)(b1 - b0), o = (size_t)b0;
    FM_CUDA(cudaMemcpyAsync(h->st_onehot + o * N * 5, onehot_host + o * N * 5, n * N * 5 * sizeof(float), cudaMemcpyHostToDevice, ls));
    DevParams p = h->p;
    FmOutputs dev = h->st_out;
    set_outputs(p, &dev);
    p.act_idx = nullptr; p.act_onehot = h->st_onehot; p.reset_mask = nullptr;
    p.env_begin = b0; p.env_end = b1;
    rc = prefetch_before_step(h, p, ls, terminal);
    if (rc) return rc;
    FM_CUDA(fm::launch_step(p, ls, false));
    h->launches += 1;
    if (terminal && h->p.auto_reset) { rc = prefetch_after_reset(h, ls, lane, b0, b1); if (rc) return rc; }
    if (out_host) {
      const size_t F = h->p.feat_global ? fm::NODE_F_GLOBAL : fm::NODE_F;
      auto d2h = [&](void* dst, const void* src, size_t per_env) -> cudaError_t {
        return dst ? cudaMemcpyAsync((char*)dst + o * per_env, (const char*)src + o * per_env, n * per_env, cudaMemcpyDeviceToHost, ls) : cudaSuccess;
      };
      FM_CUDA(d2h(out_host->node_obs, h->st_out.node_obs, N * E * F * 4));
      FM_CUDA(d2h(out_host->adj, h->st_out.adj, E * E * 4));
      FM_CUDA(d2h(out_host->obs, h->st_out.obs, N * fm::OBS_F * 4));
      FM_CUDA(d2h(out_host->reward, h->st_out.reward, N * 4));
      FM_CUDA(d2h(out_host->done, h->st_out.done, N));
      FM_CUDA(d2h(out_host->info, h->st_out.info, N * fm::INFO_F * 4));
    }
  }
  if (lane > 0) FM_CUDA(cudaEventRecord(h->lane_join[lane], ls));
  if (lane == num_lanes - 1) {
    for (int k = 1; k < num_lanes; ++k) FM_CUDA(cudaStreamWaitEvent(user, h->lane_join[k], 0));
    advance_phase(h, terminal);
    FM_CUDA(cudaStreamSynchronize(user));
  }
  return FM_OK;
}

int fm_read_info_host(FmHandle* h, float* info_host, void* stream) {
  if (!h || !info_host) return fail(FM_ERR_INVALID_ARG, "fm_read_info_host: null argument");
  int rc = use_device(h->device);
  if (rc) return rc;
  rc = ensure_staging(h);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  FM_CUDA(cudaMemcpyAsync(info_host, h->st_out.info, (size_t)h->p.B * h->p.N * fm::INFO_F * 4, cudaMemcpyDeviceToHost, st));
  FM_CUDA(cudaStreamSynchronize(st));
  return FM_OK;
}

int fm_reset_host(FmHandle* h, const uint8_t* mask_host, const FmOutputs* out_host, void* stream) {
  if (!h) return fail(FM_ERR_INVALID_ARG, "fm_reset_host: null handle");
  int rc = use_device(h->device);
  if (rc) return rc;
  rc = ensure_staging(h);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (mask_host) FM_CUDA(cudaMemcpyAsync(h->st_mask, mask_host, (size_t)h->p.B, cudaMemcpyHostToDevice, st));
  FmOutputs dev = h->st_out;
  dev.reward = nullptr; dev.done = nullptr; dev.info = nullptr;
  rc = fm_reset(h, mask_host ? h->st_mask : nullptr, &dev, stream);
  if (rc) return rc;
  rc = copy_outputs_to_host(h, out_host, false, st);
  if (rc) return rc;
  FM_CUDA(cudaStreamSynchronize(st));
  return FM_OK;
}

int fm_set_state(FmHandle* h, const FmState* st, void* stream) {
  if (!h || !st) return fail(FM_ERR_INVALID_ARG, "fm_set_state: null argument");
  int rc = use_device(h->device);
  if (rc) return rc;
  FM_CUDA(fm::launch_state_io(h->p, *st, 1, (cudaStream_t)stream));
  h->launches += 1;
  if (st->step || st->episode) h->lockstep = 0;      // the host no longer knows the episode phase of every env
  if (st->landmark_pos || st->obstacle_pos || st->wall_axis || st->wall_orient) {   // cached static distances follow the positions
    FM_CUDA(fm::launch_static_dists(h->p, (cudaStream_t)stream));
    h->launches += 1;
  }
  return FM_OK;
}

int fm_get_state(FmHandle* h, const FmState* st, void* stream) {
  if (!h || !st) return fail(FM_ERR_INVALID_ARG, "fm_get_state: null argument");
  int rc = use_device(h->device);
  if (rc) return rc;
  FM_CUDA(fm::launch_state_io(h->p, *st, 0, (cudaStream_t)stream));
  h->launches += 1;
  return FM_OK;
}

int fm_assign_costs(int device, const double* costs, int32_t num, int32_t n, int32_t* out, void* stream) {
  if (num != 0 && (!costs || !out)) return fail(FM_ERR_INVALID_ARG, "fm_assign_costs: null argument");
  if (n < 1 || n > FM_MAX_AGENTS) return fail(FM_ERR_INVALID_ARG, "fm_assign_costs: n must be in 1..%d (got %d)", FM_MAX_AGENTS, n);
  if (num < 0) return fail(FM_ERR_INVALID_ARG, "fm_assign_costs: num < 0");
  int rc = use_device(device);
  if (rc) return rc;
  FM_CUDA(fm::launch_assign(costs, nullptr, nullptr, num, n, out, (cudaStream_t)stream));
  return FM_OK;
}

int fm_assign_positions(int device, const float* agent_pos, const float* goal_pos, int32_t num, int32_t n,
                        int32_t* out, void* stream) {
  if (num != 0 && (!agent_pos || !goal_pos || !out)) return fail(FM_ERR_INVALID_ARG, "fm_assign_positions: null argument");
  if (n < 1 || n > FM_MAX_AGENTS) return fail(FM_ERR_INVALID_ARG, "fm_assign_positions: n must be in 1..%d (got %d)", FM_MAX_AGENTS, n);
  if (num < 0) return fail(FM_ERR_INVALID_ARG, "fm_assign_positions: num < 0");
  int rc = use_device(device);
  if (rc) return rc;
  FM_CUDA(fm::launch_assign(nullptr, agent_pos, goal_pos, num, n, out, (cudaStream_t)stream));
  return FM_OK;
}

int fm_assign_min_sum_costs(int device, const double* costs, int32_t num, int32_t n, int32_t* out, void* stream) {
  if (num != 0 && (!costs || !out)) return fail(FM_ERR_INVALID_ARG, "fm_assign_min_sum_costs: null argument");
  if (n < 1 || n > FM_MAX_AGENTS) return fail(FM_ERR_INVALID_ARG, "fm_assign_min_sum_costs: n must be in 1..%d (got %d)", FM_MAX_AGENTS, n);
  if (num < 0) return fail(FM_ERR_INVALID_ARG, "fm_assign_min_sum_costs: num < 0");
  int rc = use_device(device);
  if (rc) return rc;
  FM_CUDA(fm::launch_lsap(costs, nullptr, nullptr, num, n, out, (cudaStream_t)stream));
  return FM_OK;
}

int fm_assign_min_sum_positions(int device, const float* agent_pos, const float* goal_pos, int32_t num, int32_t n,
                                int32_t* out, void* stream) {
  if (num != 0 && (!agent_pos || !goal_pos || !out)) return fail(FM_ERR_INVALID_ARG, "fm_assign_min_sum_positions: null argument");
  if (n < 1 || n > FM_MAX_AGENTS) return fail(FM_ERR_INVALID_ARG, "fm_assign_min_sum_positions: n must be in 1..%d (got %d)", FM_MAX_AGENTS, n);
  if (num < 0) return fail(FM_ERR_INVALID_ARG, "fm_assign_min_sum_positions: num < 0");
  int rc = use_device(device);
  if (rc) return rc;
  FM_CUDA(fm::launch_lsap(nullptr, agent_pos, goal_pos, num, n, out, (cudaStream_t)stream));
  return FM_OK;
}

int fm_pair_dist(int device, const float* a, const float* b, int64_t num, double* out, void* stream) {
  if (!a || !b || !out) return fail(FM_ERR_INVALID_ARG, "fm_pair_dist: null argument");
  if (num < 0) return fail(FM_ERR_INVALID_ARG, "fm_pair_dist: num < 0");
  int rc = use_device(device);
  if (rc) return rc;
  FM_CUDA(fm::launch_pair_dist(a, b, (long long)num, out, (cudaStream_t)stream));
  return FM_OK;
}

int fm_edge_list(int device, const float* adj, int32_t num_graphs, int32_t E, double max_edge_dist, int32_t inclusive,
                 int32_t repeat, int64_t capacity, int64_t* graph_offsets, int64_t* edge_index, float* edge_attr,
                 int64_t* nnz_out, void* stream) {
  if (!graph_offsets || !edge_index || !edge_attr) return fail(FM_ERR_INVALID_ARG, "fm_edge_list: null output");
  if (num_graphs < 0 || E < 1 || repeat < 1 || capacity < 0) return fail(FM_ERR_INVALID_ARG, "fm_edge_list: bad sizes");
  if (num_graphs > 0 && !adj) return fail(FM_ERR_INVALID_ARG, "fm_edge_list: null adj");
  int rc = use_device(device);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  void* scratch = nullptr;
  cudaError_t e;
  // Three bit-identical forms (tests run all of them).  FM_EDGE_FORM = stream (default: count / offsets / persistent emission
  // with the next graph's loads in flight, fm_edges.cu) | three (count / one-block scan / emit, fm_kernels.cu) | fused (single
  // pass with a look-back, fm_edges.cu; FM_EDGE_FUSED=1 selects it too).  Measured at config 3: profiles/r02_j_*, r02_es_*.
  const char* form_env = getenv("FM_EDGE_FORM");          // read per call (tests flip it); ~50 ns beside three launches
  const char* fused_env = getenv("FM_EDGE_FUSED");
  int form = 0;                                           // 0 stream, 1 three, 2 fused
  if (form_env && form_env[0]) form = form_env[0] == 't' ? 1 : (form_env[0] == 'f' ? 2 : 0);
  else if (fused_env && fused_env[0] == '1') form = 2;
  if (form == 2 && fm::edge_fused_smem(E) > 96 * 1024) form = 0;
  if (form == 0 && E > 100) form = 1;                      // the streamed emission divides by E with a 20-bit reciprocal
  if (form == 2) {
    // adj read once, look-back scan; scratch = one status word per CTA + the tile counter
    FM_CUDA(cudaMallocAsync(&scratch, fm::edge_fused_scratch_bytes(num_graphs), st));
    e = fm::launch_edge_list_fused(adj, num_graphs, E, (float)max_edge_dist, inclusive, repeat, (long long)capacity, scratch,
                                   (long long*)graph_offsets, (long long*)edge_index, edge_attr, (long long*)nnz_out, st);
  } else if (form == 0) {
    // scratch: the tile sums followed by the per-graph counts (int32)
    FM_CUDA(cudaMallocAsync(&scratch, fm::edge_stream_scratch_bytes(num_graphs), st));
    e = fm::launch_edge_list_stream(adj, num_graphs, E, (float)max_edge_dist, inclusive, repeat, (long long)capacity, scratch,
                                    (long long*)graph_offsets, (long long*)edge_index, edge_attr, (long long*)nnz_out, st);
  } else {
    // count / scan / emit (fm_kernels.cu); scratch: per-CTA sums / offsets (int64) followed by the per-graph counts (int32)
    const int nb = fm::edge_list_blocks(num_graphs);
    const size_t bs_bytes = sizeof(long long) * (size_t)(nb > 0 ? nb : 1);
    FM_CUDA(cudaMallocAsync(&scratch, bs_bytes + sizeof(int) * (size_t)(num_graphs > 0 ? num_graphs : 1), st));
    long long* blocksums = (long long*)scratch;
    int* counts = (int*)((char*)scratch + bs_bytes);
    e = fm::launch_edge_list(adj, num_graphs, E, (float)max_edge_dist, inclusive, repeat, (long long)capacity,
                             counts, blocksums, (long long*)graph_offsets, (long long*)edge_index, edge_attr,
                             (long long*)nnz_out, st);
  }
  cudaFreeAsync(scratch, st);
  if (e != cudaSuccess) return fail(FM_ERR_CUDA, "fm_edge_list: %s", cudaGetErrorString(e));
  return FM_OK;
}

int fm_stats_read(FmHandle* h, double* out_dev, int32_t clear, void* stream) {
  if (!h || !out_dev) return fail(FM_ERR_INVALID_ARG, "fm_stats_read: null argument");
  int rc = use_device(h->device);
  if (rc) return rc;
  FM_CUDA(fm::launch_stats_reduce(h->stats, h->stats_rows, h->K, out_dev, clear, (cudaStream_t)stream));
  h->launches += 1;
  return FM_OK;
}

int fm_num_entities(const FmHandle* h) { return h ? h->p.E : 0; }
int fm_mapping(const FmHandle* h) { return h ? h->p.mapping + 1 : 0; }

int64_t fm_algorithmic_bytes_per_step(const FmHandle* h) {
  if (!h) return 0;
  const int64_t N = h->p.N, O = h->p.O, E = h->p.E, W = h->p.W;
  const int64_t nf = h->p.feat_global ? fm::NODE_F_GLOBAL : fm::NODE_F;
  const int64_t walls = W > 0 ? 2 * W + 1 : 0;                               // reads of wall axis / orientation / half-length
  return (30 * N + 2 * O + 5 + walls + nf * N * E + E * E) * 4 * (int64_t)h->p.B;   // SURVEY.md section 8(d), E = 2N + O + W
}

int fm_kernel_launches(const FmHandle* h, int64_t* out) {
  if (!h || !out) return fail(FM_ERR_INVALID_ARG, "fm_kernel_launches: null argument");
  *out = h->launches;
  return FM_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Formation family (include/fairmarl.h, fm_formation.cu).
struct FmFormation {
  FmFormationConfig cfg;
  int device;
  fm::FormParams p;
  void* block;
  size_t field_bytes[23];
  fm::FormAsync async;       // side stream + fork / join events of the pending-reset prefetch (split step path)
  bool has_async;
  cudaStream_t lane_stream;  // second env-range lane of fm_formation_step_many (created on first use)
  cudaEvent_t lane_fork, lane_join;
  fm::FormAsync lane_async;  // the second lane's own prefetch stream / events
  bool has_lane;
  double* stats;             // episode statistics (allocated on first fm_formation_stats_enable): [ceil(B / 32)][K] partial
  float* stats_info;         // sums, followed by [B, N, 14] info rows for the steps whose caller passes no info array
  int stats_rows, K;
};

// the 23 members of FmFormationState, in declaration order: (words per env, element size)
static void formation_fields(int N, int O, int W, size_t B, size_t (&bytes)[23]) {
  const size_t n = (size_t)N, o = (size_t)O, w = (size_t)W;
  const size_t words[23] = {2 * n, 2 * n, n, 2 * n, 2 * o, n, n, n, n, n, n, 1, 1, 1, n, 1, n, n, n, n, w, w, (size_t)(W ? 1 : 0)};
  for (int k = 0; k < 23; ++k) bytes[k] = words[k] * B * (k == 16 ? 1 : 4);      // status is uint8
}

int fm_formation_create(const FmFormationConfig* cfg, int device, FmFormation** out) {
  if (!cfg || !out) return fail(FM_ERR_INVALID_ARG, "fm_formation_create: null argument");
  *out = nullptr;
  if (cfg->num_envs <= 0) return fail(FM_ERR_INVALID_ARG, "fm_formation_create: num_envs must be > 0 (got %d)", cfg->num_envs);
  if (cfg->num_agents < 2 || cfg->num_agents > fm::formation_max_agents())
    return fail(FM_ERR_UNSUPPORTED, "fm_formation_create: num_agents must be 2..%d (got %d): the observation needs a second goal",
                fm::formation_max_agents(), cfg->num_agents);
  if (cfg->assignment < 0 || cfg->assignment > 2) return fail(FM_ERR_INVALID_ARG, "fm_formation_create: assignment must be 0 (fair), 1 (optimal) or 2 (random)");
  if (cfg->assignment != 0 && cfg->fairness_reward)
    return fail(FM_ERR_INVALID_ARG, "fm_formation_create: the base formation scenarios (optimal / random assignment) have no fairness term");
  if (cfg->num_obstacles < 0 || cfg->num_obstacles > FM_FORMATION_MAX_OBSTACLES)
    return fail(FM_ERR_INVALID_ARG, "fm_formation_create: num_obstacles must be in 0..%d (got %d)", FM_FORMATION_MAX_OBSTACLES, cfg->num_obstacles);
  if (cfg->episode_length < 1) return fail(FM_ERR_INVALID_ARG, "fm_formation_create: episode_length must be >= 1");
  if (cfg->num_walls < 0 || cfg->num_walls > 2)
    return fail(FM_ERR_INVALID_ARG, "fm_formation_create: num_walls must be 0..2 (wall_axis has two entries, :304; got %d)", cfg->num_walls);
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return fail(FM_ERR_NO_DEVICE, "fm_formation_create: no CUDA device (there is no CPU path)");
  if (device < 0 || device >= count) return fail(FM_ERR_INVALID_ARG, "fm_formation_create: device %d out of range (%d devices)", device, count);
  if (int rc = use_device(device)) return rc;
  FmFormation* h = new (std::nothrow) FmFormation();
  if (!h) return fail(FM_ERR_CUDA, "fm_formation_create: out of host memory");
  h->cfg = *cfg; h->device = device; h->has_lane = false;
  h->stats = nullptr; h->stats_info = nullptr; h->stats_rows = (cfg->num_envs + 31) / 32; h->K = fm_stats_len(cfg->num_agents);
  fm::FormParams& p = h->p;
  memset(&p, 0, sizeof(p));
  p.B = cfg->num_envs; p.N = cfg->num_agents; p.O = cfg->num_obstacles; p.episode_length = cfg->episode_length;
  p.fairness_reward = cfg->fairness_reward; p.collaborative = cfg->collaborative; p.auto_reset = cfg->auto_reset;
  p.has_max_speed = cfg->max_speed > 0.0; p.env_offset = cfg->env_offset;
  p.assignment = cfg->assignment; p.info_every_step = cfg->info_every_step; p.W = cfg->num_walls;
  p.seed_lo = (uint32_t)(cfg->seed & 0xffffffffull); p.seed_hi = (uint32_t)(cfg->seed >> 32);
  p.world_size = cfg->world_size; p.max_speed = cfg->max_speed; p.collision_rew = cfg->collision_rew; p.goal_rew = cfg->goal_rew;
  p.min_dist_thresh = cfg->min_dist_thresh; p.min_obs_dist = cfg->min_obs_dist; p.fair_rew = cfg->fair_rew; p.zeroshift = cfg->zeroshift;
  formation_fields(p.N, p.O, p.W, (size_t)p.B, h->field_bytes);
  size_t total = 0;
  for (int k = 0; k < 23; ++k) total += (h->field_bytes[k] + 255) & ~(size_t)255;
  const size_t state_bytes = total;
  total += fm::formation_recipe_floats(p.N, p.O, p.B) * sizeof(float);               // recipes of the split step path
  const size_t ready_off = total;
  total += (2 * ((size_t)(p.B + 31) / 32) * sizeof(int) + 255) & ~(size_t)255;     // logic -> image flags (two per 32-env tile) of the split step path
  const size_t pend_off = total;
  const size_t pend_bytes = fm::formation_pending_floats(p.N, p.O, p.B) * sizeof(float);   // pending resets of the split step path
  total += pend_bytes;
  cudaError_t e = cudaMalloc(&h->block, total);
  if (e != cudaSuccess) { delete h; return fail(FM_ERR_CUDA, "fm_formation_create: cudaMalloc(%zu B): %s", total, cudaGetErrorString(e)); }
  cudaMemset(h->block, 0, total);
  char* q = (char*)h->block;
  void** member = reinterpret_cast<void**>(&p.st);                                 // 23 pointers, declaration order
  for (int k = 0; k < 23; ++k) { member[k] = q; q += (h->field_bytes[k] + 255) & ~(size_t)255; }
  p.rec = reinterpret_cast<float*>((char*)h->block + state_bytes);
  const char* fused = getenv("FM_FORM_FUSED");
  p.fused = fused && fused[0] == '1';
  p.Bp = ((p.B + 31) / 32) * 32;
  h->has_async = false;
  const char* nopdl = getenv("FM_FORM_PDL");                                       // FM_FORM_PDL=0: plain stream order (A-B)
  const char* nopf = getenv("FM_FORM_PREFETCH");                                   // FM_FORM_PREFETCH=0: every reset drawn inline (A-B)
  const bool split = p.N <= 4 && p.O <= 3 && p.W == 0 && !p.fused;
  if (split && !(nopdl && nopdl[0] == '0'))
    p.ready = reinterpret_cast<int*>((char*)h->block + ready_off);                  // zeroed with the block
  if (split && !(nopf && nopf[0] == '0')) {
    p.pend = reinterpret_cast<float*>((char*)h->block + pend_off);
    cudaMemset(p.pend, 0xff, pend_bytes);                                          // tag -1: no block drawn yet
    bool ok = cudaStreamCreateWithFlags(&h->async.side, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->async.fork, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->async.join, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) { cudaFree(h->block); delete h; return fail(FM_ERR_CUDA, "fm_formation_create: side stream / events: %s", cudaGetErrorString(cudaGetLastError())); }
    h->has_async = true;
  }
  *out = h;
  return FM_OK;
}

int fm_formation_destroy(FmFormation* h) {
  if (!h) return FM_OK;
  if (int rc = use_device(h->device)) return rc;
  cudaDeviceSynchronize();
  if (h->has_async) { cudaEventDestroy(h->async.fork); cudaEventDestroy(h->async.join); cudaStreamDestroy(h->async.side); }
  if (h->has_lane) {
    cudaEventDestroy(h->lane_fork); cudaEventDestroy(h->lane_join); cudaStreamDestroy(h->lane_stream);
    if (h->has_async) { cudaEventDestroy(h->lane_async.fork); cudaEventDestroy(h->lane_async.join); cudaStreamDestroy(h->lane_async.side); }
  }
  cudaFree(h->stats);
  cudaFree(h->block);
  delete h;
  return FM_OK;
}

int fm_formation_reset(FmFormation* h, const uint8_t* mask, const FmOutputs* out, void* stream) {
  if (!h || !out) return fail(FM_ERR_INVALID_ARG, "fm_formation_reset: null argument");
  if (int rc = use_device(h->device)) return rc;
  fm::FormParams p = h->p;
  p.out = *out; p.mask = mask; p.actions = nullptr;
  FM_CUDA(fm::launch_formation(p, true, (cudaStream_t)stream));
  return FM_OK;
}

// The step's outputs: with statistics on, info rows always go somewhere (the handle's own rows when the caller passes none),
// so that the statistics do not depend on which outputs the caller asks for.
static FmOutputs formation_outputs(const FmFormation* h, const FmOutputs& out) {
  FmOutputs o = out;
  if (h->p.stats && !o.info) o.info = h->stats_info;
  return o;
}

int fm_formation_step(FmFormation* h, const int32_t* actions, const FmOutputs* out, void* stream) {
  if (!h || !actions || !out) return fail(FM_ERR_INVALID_ARG, "fm_formation_step: null argument");
  if (int rc = use_device(h->device)) return rc;
  fm::FormParams p = h->p;
  p.out = formation_outputs(h, *out); p.actions = actions; p.mask = nullptr;
  FM_CUDA(fm::launch_formation(p, false, (cudaStream_t)stream, h->has_async ? &h->async : nullptr));
  return FM_OK;
}

// The handle's launch parameters restricted to envs [start, start + count) (start a multiple of 32): every per-env pointer
// moves by its own stride, the Philox key by `start`; tile-indexed blocks (recipes, ready flags, statistics rows) by whole tiles.
static fm::FormParams formation_slice(const FmFormation* h, int start, int count, const FmOutputs& out, const int32_t* actions) {
  fm::FormParams p = h->p;
  const size_t B = (size_t)h->p.B;
  void** member = reinterpret_cast<void**>(&p.st);
  for (int k = 0; k < 23; ++k)
    if (member[k]) member[k] = (char*)member[k] + h->field_bytes[k] / B * (size_t)start;
  const size_t N = (size_t)p.N, E = 2 * N + (size_t)p.O + (size_t)p.W;
  p.out = formation_outputs(h, out);
  if (p.out.obs) p.out.obs += (size_t)start * N * FM_FORMATION_OBS_DIM;
  if (p.out.node_obs) p.out.node_obs += (size_t)start * N * E * FM_FORMATION_NODE_FEAT_DIM;
  if (p.out.adj) p.out.adj += (size_t)start * E * E;
  if (p.out.reward) p.out.reward += (size_t)start * N;
  if (p.out.done) p.out.done += (size_t)start * N;
  if (p.out.info) p.out.info += (size_t)start * N * FM_INFO_DIM;
  p.actions = actions + (size_t)start * N;
  p.mask = nullptr;
  p.env_offset += start;
  p.B = count;
  if (p.rec) p.rec += fm::formation_recipe_floats(p.N, p.O, start);
  if (p.ready) p.ready += 2 * (start / 32);
  if (p.pend) p.pend += start;                          // SoA: the field stride stays the handle's Bp
  if (p.stats) p.stats += (size_t)(start / 32) * h->K;
  return p;
}

int fm_formation_step_many(FmFormation* h, const int32_t* actions, int32_t T, const FmOutputs* outs, void* stream) {
  if (!h || !actions || !outs) return fail(FM_ERR_INVALID_ARG, "fm_formation_step_many: null argument");
  if (T < 0) return fail(FM_ERR_INVALID_ARG, "fm_formation_step_many: T must be >= 0");
  if (int rc = use_device(h->device)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int B = h->p.B;
  // One lane by default: two env-range lanes on two streams (FM_FORM_LANES=2) are bit-identical but measured 3 % slower
  // (66.9 vs 65.0 us / step at 65 536 envs, profiles/r02_q) -- the logic kernels of both lanes fill the register file
  // (16 warps x 128 registers per SM), so the other lane's image kernel finds no room to run beside them.
  const char* lanes_env = getenv("FM_FORM_LANES");
  const bool two = B >= 4096 && lanes_env && lanes_env[0] == '2';
  if (two && !h->has_lane) {
    bool ok = cudaStreamCreateWithFlags(&h->lane_stream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->lane_fork, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->lane_join, cudaEventDisableTiming) == cudaSuccess;
    if (h->has_async) {
      ok = ok && cudaStreamCreateWithFlags(&h->lane_async.side, cudaStreamNonBlocking) == cudaSuccess;
      ok = ok && cudaEventCreateWithFlags(&h->lane_async.fork, cudaEventDisableTiming) == cudaSuccess;
      ok = ok && cudaEventCreateWithFlags(&h->lane_async.join, cudaEventDisableTiming) == cudaSuccess;
    }
    if (!ok) return fail(FM_ERR_CUDA, "fm_formation_step_many: lane stream / events: %s", cudaGetErrorString(cudaGetLastError()));
    h->has_lane = true;
  }
  const int half = two ? ((B / 2 + 31) / 32) * 32 : B;
  if (two) { FM_CUDA(cudaEventRecord(h->lane_fork, st)); FM_CUDA(cudaStreamWaitEvent(h->lane_stream, h->lane_fork, 0)); }
  const size_t step_actions = (size_t)B * h->p.N;
  for (int t = 0; t < T; ++t) {
    const int32_t* a = actions + (size_t)t * step_actions;
    FM_CUDA(fm::launch_formation(formation_slice(h, 0, half, outs[t], a), false, st, h->has_async ? &h->async : nullptr));
    if (two) FM_CUDA(fm::launch_formation(formation_slice(h, half, B - half, outs[t], a), false, h->lane_stream, h->has_async ? &h->lane_async : nullptr));
  }
  if (two) { FM_CUDA(cudaEventRecord(h->lane_join, h->lane_stream)); FM_CUDA(cudaStreamWaitEvent(st, h->lane_join, 0)); }
  return FM_OK;
}

static int formation_state_copy(FmFormation* h, const FmFormationState* st, bool to_handle, void* stream, const char* who) {
  if (!h || !st) return fail(FM_ERR_INVALID_ARG, "%s: null argument", who);
  if (int rc = use_device(h->device)) return rc;
  void* const* mine = reinterpret_cast<void* const*>(&h->p.st);
  void* const* theirs = reinterpret_cast<void* const*>(st);
  for (int k = 0; k < 23; ++k) {
    if (!theirs[k] || h->field_bytes[k] == 0) continue;
    FM_CUDA(cudaMemcpyAsync(to_handle ? mine[k] : theirs[k], to_handle ? theirs[k] : mine[k], h->field_bytes[k],
                            cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  }
  return FM_OK;
}

int fm_formation_set_state(FmFormation* h, const FmFormationState* st, void* stream) {
  return formation_state_copy(h, st, true, stream, "fm_formation_set_state");
}

int fm_formation_get_state(FmFormation* h, const FmFormationState* st, void* stream) {
  return formation_state_copy(h, st, false, stream, "fm_formation_get_state");
}

int fm_formation_stats_enable(FmFormation* h, int32_t enable, void* stream) {
  if (!h) return fail(FM_ERR_INVALID_ARG, "fm_formation_stats_enable: null argument");
  if (int rc = use_device(h->device)) return rc;
  if (enable && !h->stats) {
    const size_t rows = (size_t)h->stats_rows * h->K * sizeof(double);
    const size_t info = (size_t)h->p.B * h->p.N * FM_INFO_DIM * sizeof(float);
    void* block = nullptr;
    FM_CUDA(cudaMalloc(&block, rows + info));
    cudaError_t e = cudaMemsetAsync(block, 0, rows + info, (cudaStream_t)stream);
    if (e != cudaSuccess) { cudaFree(block); return fail(FM_ERR_CUDA, "fm_formation_stats_enable: %s", cudaGetErrorString(e)); }
    h->stats = (double*)block;
    h->stats_info = (float*)((char*)block + rows);
  }
  h->p.stats = enable ? h->stats : nullptr;
  return FM_OK;
}

int fm_formation_stats_read(FmFormation* h, double* out_dev, int32_t clear, void* stream) {
  if (!h || !out_dev) return fail(FM_ERR_INVALID_ARG, "fm_formation_stats_read: null argument");
  if (!h->p.stats) return fail(FM_ERR_INVALID_ARG, "fm_formation_stats_read: episode statistics are off (fm_formation_stats_enable)");
  if (int rc = use_device(h->device)) return rc;
  FM_CUDA(fm::launch_stats_reduce(h->stats, h->stats_rows, h->K, out_dev, clear, (cudaStream_t)stream));
  return FM_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Fused graph-network forward (fm_policy.cu).
int64_t fm_gnn_weight_floats(const FmGnnConfig* cfg) {
  if (!cfg) return 0;
  return fm::gnn_weight_count(cfg->embed_layers, cfg->conv_layers);
}

int fm_gnn_supported(int32_t num_entities, int32_t node_feat_dim) {
  return fm::gnn_supported_entities(num_entities) && node_feat_dim >= 2 && node_feat_dim <= 17 ? 1 : 0;
}

int fm_gnn_mapping(int32_t num_entities, int32_t node_feat_dim) {
  if (node_feat_dim < 2 || node_feat_dim > 17) return 0;
  if (fm::gnn_supported_entities(num_entities)) return 1;
  return fm::gnn_wide_supported_entities(num_entities) ? 2 : 0;
}

int fm_gnn_forward(int device, const FmGnnConfig* cfg, const float* weights, const float* node_obs, const float* adj,
                   const int32_t* agent_id, float* out, void* stream) {
  if (!cfg || !weights || !node_obs || !adj || !out) return fail(FM_ERR_INVALID_ARG, "fm_gnn_forward: null argument");
  if (cfg->num_graphs < 0 || cfg->graphs_per_adj < 1) return fail(FM_ERR_INVALID_ARG, "fm_gnn_forward: bad graph counts");
  if (cfg->mapping < 0 || cfg->mapping > 2)
    return fail(FM_ERR_INVALID_ARG, "fm_gnn_forward: mapping %d (0 auto, 1 warp per graph, 2 CTA per graph)", cfg->mapping);
  const int E = cfg->num_entities, NF = cfg->node_feat_dim;
  const bool ok = cfg->mapping == 0 ? fm_gnn_mapping(E, NF) != 0
                : cfg->mapping == 1 ? fm_gnn_supported(E, NF) != 0
                                    : fm::gnn_wide_supported_entities(E) && NF >= 2 && NF <= 17;
  if (!ok)
    return fail(FM_ERR_UNSUPPORTED, "fm_gnn_forward: mapping %d is not available for %d entities x %d features", cfg->mapping, E, NF);
  if (cfg->embed_layers < 0 || cfg->embed_layers > 2 || cfg->conv_layers < 1 || cfg->conv_layers > 8 || cfg->aggr < 0 || cfg->aggr > 3)
    return fail(FM_ERR_UNSUPPORTED, "fm_gnn_forward: embed_layers %d / conv_layers %d / aggr %d", cfg->embed_layers, cfg->conv_layers, cfg->aggr);
  int rc = use_device(device);
  if (rc) return rc;
  FM_CUDA(fm::launch_gnn(*cfg, weights, node_obs, adj, agent_id, out, 0, (cudaStream_t)stream));
  return FM_OK;
}

int fm_gnn_gather(int device, const FmGnnConfig* cfg, int32_t k, const float* weights, const float* node_obs,
                  const float* adj, const int32_t* agent_id, float* out, void* stream) {
  if (!cfg || !weights || !node_obs || !adj || !agent_id || !out) return fail(FM_ERR_INVALID_ARG, "fm_gnn_gather: null argument");
  if (cfg->aggr != 0) return fail(FM_ERR_INVALID_ARG, "fm_gnn_gather: aggr %d (the gather is a node aggregation: 0)", cfg->aggr);
  if (k < 1 || k > cfg->num_entities)
    return fail(FM_ERR_INVALID_ARG, "fm_gnn_gather: k %d nodes per graph (1..%d)", k, cfg->num_entities);
  if (cfg->num_graphs < 0 || cfg->graphs_per_adj < 1) return fail(FM_ERR_INVALID_ARG, "fm_gnn_gather: bad graph counts");
  if (cfg->mapping < 0 || cfg->mapping > 2)
    return fail(FM_ERR_INVALID_ARG, "fm_gnn_gather: mapping %d (0 auto, 1 warp per graph, 2 CTA per graph)", cfg->mapping);
  const int E = cfg->num_entities, NF = cfg->node_feat_dim;
  const bool ok = cfg->mapping == 0 ? fm_gnn_mapping(E, NF) != 0
                : cfg->mapping == 1 ? fm_gnn_supported(E, NF) != 0
                                    : fm::gnn_wide_supported_entities(E) && NF >= 2 && NF <= 17;
  if (!ok)
    return fail(FM_ERR_UNSUPPORTED, "fm_gnn_gather: mapping %d is not available for %d entities x %d features", cfg->mapping, E, NF);
  if (cfg->embed_layers < 0 || cfg->embed_layers > 2 || cfg->conv_layers < 1 || cfg->conv_layers > 8)
    return fail(FM_ERR_UNSUPPORTED, "fm_gnn_gather: embed_layers %d / conv_layers %d", cfg->embed_layers, cfg->conv_layers);
  int rc = use_device(device);
  if (rc) return rc;
  FM_CUDA(fm::launch_gnn(*cfg, weights, node_obs, adj, agent_id, out, k, (cudaStream_t)stream));
  return FM_OK;
}

int64_t fm_head_weight_floats(const FmHeadConfig* cfg) {
  if (!cfg) return 0;
  return fm::head_weight_count(cfg->layers, cfg->recurrent);
}

int fm_policy_head(int device, const FmHeadConfig* cfg, const float* weights, const float* obs, const float* nbd,
                   const float* rnn_in, const float* mask, const float* u, float* rnn_out, float* logp, int64_t* action,
                   float* value, void* stream) {
  if (!cfg || !weights || !nbd) return fail(FM_ERR_INVALID_ARG, "fm_policy_head: null argument");
  if (cfg->obs_dim < 0 || cfg->obs_dim > 16 || (cfg->obs_dim > 0 && !obs)) return fail(FM_ERR_INVALID_ARG, "fm_policy_head: obs_dim must be 0..16 (with obs)");
  if (cfg->layers < 0 || cfg->layers > 2 || cfg->num_outputs < 1 || cfg->num_outputs > 8) return fail(FM_ERR_UNSUPPORTED, "fm_policy_head: layers %d / outputs %d", cfg->layers, cfg->num_outputs);
  if (cfg->recurrent && (!rnn_in || !mask || !rnn_out)) return fail(FM_ERR_INVALID_ARG, "fm_policy_head: recurrent head needs rnn_in, mask, rnn_out");
  if (!value && (!logp || !action)) return fail(FM_ERR_INVALID_ARG, "fm_policy_head: actor head needs logp and action (or pass value for the critic)");
  int rc = use_device(device);
  if (rc) return rc;
  FM_CUDA(fm::launch_head(*cfg, weights, obs, nbd, rnn_in, mask, u, rnn_out, logp, (long long*)action, value, (cudaStream_t)stream));
  return FM_OK;
}

int64_t fm_critic_head_weight_floats(const FmCriticHeadConfig* cfg) {
  if (!cfg) return 0;
  return fm::critic_head_weight_count(cfg->cent_dim + cfg->nbd_dim, cfg->layers, cfg->recurrent);
}

int fm_critic_head(int device, const FmCriticHeadConfig* cfg, const float* weights, const float* cent_obs, const float* nbd,
                   const float* rnn_in, const float* mask, float* rnn_out, float* value, void* stream) {
  if (!cfg || !weights || !nbd || !value) return fail(FM_ERR_INVALID_ARG, "fm_critic_head: null argument");
  if (cfg->num_rows < 0 || cfg->cent_dim < 0 || cfg->nbd_dim < 1 || (cfg->cent_dim > 0 && !cent_obs))
    return fail(FM_ERR_INVALID_ARG, "fm_critic_head: num_rows %d / cent_dim %d (with cent_obs) / nbd_dim %d", cfg->num_rows,
                cfg->cent_dim, cfg->nbd_dim);
  if (cfg->cent_dim > 0 && (cfg->rows_per_env < 1 || cfg->num_rows % cfg->rows_per_env != 0))
    return fail(FM_ERR_INVALID_ARG, "fm_critic_head: %d rows are not a whole number of envs of %d rows", cfg->num_rows, cfg->rows_per_env);
  if ((int64_t)cfg->cent_dim + cfg->nbd_dim > fm::CRITIC_HEAD_MAX_IN)
    return fail(FM_ERR_UNSUPPORTED, "fm_critic_head: %lld input features (at most %d)", (long long)cfg->cent_dim + cfg->nbd_dim,
                fm::CRITIC_HEAD_MAX_IN);
  if (cfg->layers < 0 || cfg->layers > 2) return fail(FM_ERR_UNSUPPORTED, "fm_critic_head: layers %d (0..2)", cfg->layers);
  if (cfg->recurrent && (!rnn_in || !mask || !rnn_out)) return fail(FM_ERR_INVALID_ARG, "fm_critic_head: recurrent head needs rnn_in, mask, rnn_out");
  int rc = use_device(device);
  if (rc) return rc;
  FM_CUDA(fm::launch_critic_head(*cfg, weights, cent_obs, nbd, rnn_in, mask, rnn_out, value, (cudaStream_t)stream));
  return FM_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Training side of the rollout buffer (fm_buffer.cu).
static int buffer_shape(const char* fn, int32_t T, int32_t B, int32_t N) {
  if (T < 1 || B < 1 || N < 1) return fail(FM_ERR_INVALID_ARG, "%s: episode_length %d / num_envs %d / num_agents %d (each >= 1)", fn, T, B, N);
  if ((int64_t)T * B * N >= ((int64_t)1 << 31))
    return fail(FM_ERR_INVALID_ARG, "%s: T * B * N = %lld samples (at most 2^31 - 1)", fn, (long long)T * B * N);
  return FM_OK;
}

static bool norm_ok(const float* mean, const float* stdv) { return (mean == nullptr) == (stdv == nullptr); }

int fm_buffer_returns(int device, const FmReturnsConfig* cfg, const float* next_value, float* value_preds, const float* rewards,
                      const float* masks, const float* bad_masks, const float* norm_mean, const float* norm_std,
                      float* returns, void* stream) {
  if (!cfg || !next_value || !value_preds || !rewards || !masks || !returns || (cfg->use_proper_time_limits && !bad_masks))
    return fail(FM_ERR_INVALID_ARG, "fm_buffer_returns: null argument");
  if (!norm_ok(norm_mean, norm_std)) return fail(FM_ERR_INVALID_ARG, "fm_buffer_returns: norm_mean and norm_std are both given or both null");
  if (int rc = buffer_shape("fm_buffer_returns", cfg->episode_length, cfg->num_envs, cfg->num_agents)) return rc;
  if (int rc = use_device(device)) return rc;
  FM_CUDA(fm::launch_buffer_returns(*cfg, next_value, value_preds, rewards, masks, bad_masks, norm_mean, norm_std, returns,
                                    (cudaStream_t)stream));
  return FM_OK;
}

int fm_buffer_advantages(int device, int32_t episode_length, int32_t num_envs, int32_t num_agents, const float* returns,
                         const float* value_preds, const float* active_masks, const float* norm_mean, const float* norm_std,
                         float* advantages, float* stats, double* workspace, void* stream) {
  if (!returns || !value_preds || !active_masks || !advantages || !stats || !workspace)
    return fail(FM_ERR_INVALID_ARG, "fm_buffer_advantages: null argument");
  if (!norm_ok(norm_mean, norm_std)) return fail(FM_ERR_INVALID_ARG, "fm_buffer_advantages: norm_mean and norm_std are both given or both null");
  if (int rc = buffer_shape("fm_buffer_advantages", episode_length, num_envs, num_agents)) return rc;
  if (int rc = use_device(device)) return rc;
  FM_CUDA(fm::launch_buffer_advantages((long long)episode_length * num_envs * num_agents, returns, value_preds, active_masks,
                                       norm_mean, norm_std, advantages, stats, workspace, (cudaStream_t)stream));
  return FM_OK;
}

int fm_buffer_minibatch(int device, const FmMinibatchConfig* cfg, const FmBufferSlabs* in, const int64_t* perm,
                        const FmMinibatch* out, void* stream) {
  if (!cfg || !in || !perm || !out) return fail(FM_ERR_INVALID_ARG, "fm_buffer_minibatch: null argument");
  const void* const req[] = {in->obs, in->node_obs, in->adj_env, in->rnn_states, in->rnn_states_critic, in->actions,
                             in->action_log_probs, in->value_preds, in->returns, in->masks, in->active_masks, in->advantages,
                             out->share_obs, out->obs, out->node_obs, out->adj, out->agent_id, out->share_agent_id,
                             out->rnn_states, out->rnn_states_critic, out->actions, out->value_preds, out->returns, out->masks,
                             out->active_masks, out->old_action_log_probs, out->adv_targ};
  for (const void* q : req)
    if (!q) return fail(FM_ERR_INVALID_ARG, "fm_buffer_minibatch: null argument");
  const int T = cfg->episode_length, B = cfg->num_envs, N = cfg->num_agents;
  if (int rc = buffer_shape("fm_buffer_minibatch", T, B, N)) return rc;
  if (cfg->num_entities < 1 || cfg->obs_dim < 1 || cfg->node_feat_dim < 1 || cfg->rnn_floats < 1)
    return fail(FM_ERR_INVALID_ARG, "fm_buffer_minibatch: num_entities %d / obs_dim %d / node_feat_dim %d / rnn_floats %d (each >= 1)",
                cfg->num_entities, cfg->obs_dim, cfg->node_feat_dim, cfg->rnn_floats);
  const int64_t samples = (int64_t)T * B * N, K = cfg->num_mini_batch;
  int64_t units, per, rows;                      // units: what the permutation ranges over
  if (cfg->mode == FM_MINIBATCH_FEED_FORWARD) {
    units = samples;
    if (K < 1 || K > units) return fail(FM_ERR_INVALID_ARG, "fm_buffer_minibatch: num_mini_batch %lld for %lld samples", (long long)K, (long long)units);
    if (cfg->mini_batch_size < 0 || (int64_t)cfg->mini_batch_size * K > units)
      return fail(FM_ERR_INVALID_ARG, "fm_buffer_minibatch: %lld mini-batches of %d samples from %lld", (long long)K, cfg->mini_batch_size,
                  (long long)units);
    per = cfg->mini_batch_size ? cfg->mini_batch_size : units / K;
    rows = per;
  } else if (cfg->mode == FM_MINIBATCH_RECURRENT || cfg->mode == FM_MINIBATCH_NAIVE_RECURRENT) {
    if (cfg->mini_batch_size != 0) return fail(FM_ERR_INVALID_ARG, "fm_buffer_minibatch: mini_batch_size is a feed-forward option");
    const bool chunked = cfg->mode == FM_MINIBATCH_RECURRENT;
    if (chunked && cfg->data_chunk_length < 1)
      return fail(FM_ERR_INVALID_ARG, "fm_buffer_minibatch: data_chunk_length %d (>= 1)", cfg->data_chunk_length);
    units = chunked ? samples / cfg->data_chunk_length : (int64_t)B * N;
    if (K < 1 || K > units)
      return fail(FM_ERR_INVALID_ARG, "fm_buffer_minibatch: num_mini_batch %lld for %lld %s", (long long)K, (long long)units,
                  chunked ? "chunks" : "columns");
    if (!chunked && units % K != 0)   // the reference yields another number of mini-batches, or raises IndexError mid-epoch
      return fail(FM_ERR_INVALID_ARG, "fm_buffer_minibatch: %lld columns are not divisible by num_mini_batch %lld", (long long)units, (long long)K);
    per = units / K;
    rows = per * (chunked ? cfg->data_chunk_length : T);
  } else {
    return fail(FM_ERR_INVALID_ARG, "fm_buffer_minibatch: mode %d (0 feed-forward, 1 recurrent, 2 naive recurrent)", cfg->mode);
  }
  if (cfg->mini_batch < 0 || cfg->mini_batch >= K)
    return fail(FM_ERR_INVALID_ARG, "fm_buffer_minibatch: mini_batch %d of %lld", cfg->mini_batch, (long long)K);
  if (int rc = use_device(device)) return rc;
  FM_CUDA(fm::launch_buffer_minibatch(*cfg, rows, per, (int)per, cfg->mini_batch * per, *in, (const long long*)perm, *out,
                                      (cudaStream_t)stream));
  return FM_OK;
}

}  // extern "C"
