/*
 * fairmarl.h -- C ABI of the B200-native batched GraphMPE `navigation_graph` simulator.
 *
 * One shared library (libfairmarl.so), plain pointers and sizes, no torch / C++ types.
 * Every entry point states the reference interface it replaces (paths relative to the
 * Jaroan/Fair-MARL checkout).  The reference is pure Python: there is no existing FFI, so the
 * "binding a maintainer would add" is a ctypes stub (INTEGRATION.md) selected in
 * onpolicy/scripts/train_mpe.py:21-43 (make_train_env) instead of GraphSubprocVecEnv.
 *
 * Conventions
 *   - All pointers in FmState / FmOutputs / actions are DEVICE pointers unless the function name
 *     ends in _host.  Any output pointer may be NULL (= not wanted).
 *   - All calls are asynchronous on the caller-supplied stream (a cudaStream_t passed as void*),
 *     except the *_host calls, which synchronise that stream before returning.
 *   - The handle owns the internal SoA state, RNG counters and statistic accumulators; the caller
 *     owns every buffer it passes in.  A handle is bound to one device and is not thread-safe.
 *   - Return value: 0 on success, a negative FmStatus otherwise; fm_last_error() gives the text.
 *     Nothing here throws, aborts or falls back to a CPU path.
 *   - Entity order (reference World.entities, multiagent/core.py:186):
 *     agents 0..N-1, landmarks N..2N-1, obstacles 2N..2N+O-1, walls 2N+O..2N+O+W-1;  E = 2N + O + W.
 */
#ifndef FAIRMARL_H_
#define FAIRMARL_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FM_ABI_VERSION 6
#define FM_OBS_DIM 7         /* navigation_graph.py:826-857 */
#define FM_NODE_FEAT_DIM 11  /* navigation_graph.py:1079-1124 (relative features) */
#define FM_INFO_DIM 14       /* navigation_graph.py:625-647 + environment.py:857 */
#define FM_MAX_AGENTS 32

typedef enum FmStatus {
  FM_OK = 0,
  FM_ERR_INVALID_ARG = -1,
  FM_ERR_CUDA = -2,
  FM_ERR_UNSUPPORTED = -3,
  FM_ERR_NO_DEVICE = -4
} FmStatus;

/* The argparse fields Scenario.make_world reads (navigation_graph.py:94-129, :144, :188, :208).
 * Reals are double because the reference holds them as Python floats and compares float64
 * distances against them (thresholds must be the same IEEE doubles). */
typedef struct FmConfig {
  int32_t num_envs;        /* B on THIS device */
  int32_t num_agents;      /* N = num_landmarks, 1..32 */
  int32_t num_obstacles;   /* O >= 0 */
  int32_t episode_length;  /* world_length, environment.py:237-247 */
  int64_t env_offset;      /* global index of local env 0: RNG streams are keyed by global index */
  uint64_t seed;
  double world_size;       /* 2 */
  double max_speed;        /* 2; <= 0 means None (no clamp, no Min_time_to_goal) */
  double collision_rew;
  double goal_rew;
  double min_dist_thresh;
  double fair_rew;
  double zeroshift;
  double max_edge_dist;
  int32_t fairness_reward; /* 1: navigation_graph.py (FA+FR); 0: nav_graph_goalassign_noFair.py (FA) */
  int32_t collaborative;   /* environment.py:867-870 */
  int32_t auto_reset;      /* env_wrappers.py:859-865 (graphworker) */
  int32_t info_every_step; /* 0: info rows are written on terminal steps only */
  int32_t mapping;         /* kernel mapping: 0 auto (agent-warp when compiled for (N, O), else group-per-env),
                              1 group-per-env, 2 agent-warp.  Results are identical. */
  int32_t graph_feat_global; /* 0: graph_feat_type 'relative' (node_obs [B,N,E,11], navigation_graph.py:1079-1124);
                                1: 'global' (node_obs [B,N,E,7] = [vel, pos, goal, type], :1058-1077) */
  int32_t num_walls;       /* W = 0, 1 or 2 axis-aligned wall segments (navigation_graph.py:181-196, :287-324; core.py:36-55,
                              :407-462); agent-warp kernels at N = 3, O = 3 (and 4 / 2 / 1), else group-per-env; not with graph_feat_global */
  int32_t reserved_;
} FmConfig;

/* Per-step outputs, API layout (what GraphSubprocVecEnv.step_wait stacks, env_wrappers.py:988-996). */
typedef struct FmOutputs {
  float* obs;        /* [B, N, 7] */
  float* node_obs;   /* [B, N, E, 11]  ([B, N, E, 7] with graph_feat_global) */
  float* adj;        /* [B, E, E]   (identical for the N agents of an env: written once) */
  float* reward;     /* [B, N] */
  uint8_t* done;     /* [B, N] */
  float* info;       /* [B, N, 14] in FM_INFO_* order; terminal-step values survive auto-reset */
} FmOutputs;

enum {
  FM_INFO_INDIVIDUAL_REWARD = 0, FM_INFO_DIST_TO_GOAL, FM_INFO_TIME_REQ_TO_GOAL,
  FM_INFO_NUM_AGENT_COLLISIONS, FM_INFO_NUM_OBST_COLLISIONS, FM_INFO_DISTANCE_MEAN,
  FM_INFO_DISTANCE_VARIANCE, FM_INFO_MEAN_BY_VARIANCE, FM_INFO_DISTS_TRAVELED, FM_INFO_TIME_TAKEN,
  FM_INFO_TIME_MEAN, FM_INFO_TIME_STDDEV, FM_INFO_TIME_MEAN_BY_STDDEV, FM_INFO_MIN_TIME_TO_GOAL
};

/* Complete simulator state in API layout (what World + Scenario carry between steps:
 * core.py:11-20, navigation_graph.py:93, :214-225, :617-618).  NULL members are skipped. */
typedef struct FmState {
  float* pos;                      /* [B, N, 2] */
  float* vel;                      /* [B, N, 2] */
  float* p_dist;                   /* [B, N] */
  float* landmark_pos;             /* [B, N, 2] */
  float* obstacle_pos;             /* [B, O, 2] */
  int32_t* goal_match;             /* [B, N] */
  float* dists_to_goal;            /* [B, N]  (-1: not yet visited this episode) */
  float* times_required;           /* [B, N]  (-1: goal not reached) */
  float* dist_left_to_goal;        /* [B, N] */
  int32_t* num_agent_collisions;   /* [B, N] */
  int32_t* num_obstacle_collisions;/* [B, N] */
  float* dist_traveled_mean;       /* [B] */
  float* dist_traveled_stddev;     /* [B] */
  int32_t* step;                   /* [B] */
  float* min_time;                 /* [B, N] */
  int32_t* episode;                /* [B]  resets so far (RNG counter) */
  float* wall_axis;                /* [B, W]  wall.axis_pos */
  int32_t* wall_orient;            /* [B, W]  0 = 'H', 1 = 'V' */
  float* wall_len;                 /* [B]     half-length (scenario.wall_length), fixed per env */
} FmState;

typedef struct FmHandle FmHandle;

/* GraphSubprocVecEnv.__init__ + GraphMPEEnv + Scenario.make_world
 * (env_wrappers.py:951-981, MPE_env.py:55-77, navigation_graph.py:48-210). */
int fm_create(const FmConfig* cfg, int device, FmHandle** out);
/* GraphSubprocVecEnv.close (env_wrappers.py:1010-1021). */
int fm_destroy(FmHandle* h);

/* GraphSubprocVecEnv.reset -> MultiAgentGraphEnv.reset -> Scenario.reset_world/random_scenario
 * (env_wrappers.py:997-1002, environment.py:882-898, navigation_graph.py:212-570), incl. the
 * lexifair goal assignment (navigation_graph.py:555-561).  mask: uint8 [B] or NULL (= all envs).
 * Envs with mask 0 keep their state; obs / node_obs / adj of ALL envs are written to `out`. */
int fm_reset(FmHandle* h, const uint8_t* mask, const FmOutputs* out, void* stream);
/* Observation of the CURRENT state into `out` (obs, node_obs, adj) without resetting or stepping anything
 * (MultiAgentGraphEnv._get_obs / graph_observation on the live world, environment.py:882-898 minus the reset). */
int fm_observe(FmHandle* h, const FmOutputs* out, void* stream);

/* SoA observation mode: the values of fm_observe as one plane per value, envs fastest (device pointers, any may be NULL):
 *   obs [N][7][S], node_obs [N][E][F][S] (F = 11, or 7 with graph_feat_global), adj [E][E][S], S = fm_soa_stride(h) >= B
 * (a multiple of 4; planes are 16-byte aligned when the arrays are).  For device-side consumers that walk envs in lanes;
 * 16-byte loads and streaming stores throughout (csrc/fm_soa.cu).  Bit-identical to the API layout.  No walls. */
typedef struct FmSoaOutputs {
  float* obs;
  float* node_obs;
  float* adj;
} FmSoaOutputs;
int fm_soa_stride(const FmHandle* h);
int fm_observe_soa(FmHandle* h, const FmSoaOutputs* out, void* stream);

/* Non-finite guard (SURVEY.md section 5.3; core.py:392 is a latent 0/0 in the reference): flags[b] = 1 if the dynamic
 * state of env b holds a NaN / Inf (positions, velocities, travelled distances, running statistics), else 0; *count = how
 * many.  int32 device pointers, either may be NULL. */
int fm_check_finite(FmHandle* h, int32_t* flags, int32_t* count, void* stream);

/* GraphSubprocVecEnv.step -> graphworker -> MultiAgentGraphEnv.step (env_wrappers.py:983-996,
 * :856-865, environment.py:816-877): action decode, World.step (core.py:250-274), observation /
 * reward / graph_observation / done / info_callback per agent in the reference's order, and the
 * worker's auto-reset.  actions: int32 [B, N] in {0..4} (0 no-op, 1 +x, 2 -x, 3 +y, 4 -y). */
int fm_step(FmHandle* h, const int32_t* actions, const FmOutputs* out, void* stream);
/* Same, with the [B, N, 5] float one-hot (or any float 5-vector) the runner sends
 * (graph_mpe_runner.py:429-431; decode environment.py:301-311). */
int fm_step_onehot(FmHandle* h, const float* onehot, const FmOutputs* out, void* stream);

/* num_steps consecutive fm_step calls from one host call (rollout inner loop without per-step host
 * overhead): step t uses actions + t*B*N and writes outs[t].  `outs` is a HOST array of structs
 * holding DEVICE pointers. */
int fm_step_many(FmHandle* h, const int32_t* actions, int32_t num_steps, const FmOutputs* outs, void* stream);

/* Host-buffer form of fm_step_onehot: `onehot` and every member of `out` are HOST pointers
 * (pinned for full speed).  Copies actions in, steps, copies the requested outputs back and
 * synchronises `stream`.  This is the call a ShareVecEnv.step() drop-in makes. */
int fm_step_host(FmHandle* h, const float* onehot_host, const FmOutputs* out_host, void* stream);
/* The same step issued as `num_lanes` env-range lanes (1..8), one call per lane in the order 0 .. num_lanes - 1: lane k
 * covers envs [k * L, min(B, (k + 1) * L)), L = ceil(B / num_lanes) rounded up to 128; fm_host_lane_range gives the range.
 * A call enqueues its lane -- H2D of that range of `onehot_host`, the step kernel on that range, D2H of that range of every
 * output -- and returns without waiting, except the last one, which waits for all lanes.  The caller fills the action rows
 * of lane k + 1 (GMPERunner builds them as float64 one-hot, graph_mpe_runner.py:429-431: the conversion into the pinned
 * float32 buffer costs as much as a fifth of the copies) while lane k's results cross the bus.  Pointers are the FULL arrays. */
int fm_step_host_lane(FmHandle* h, const float* onehot_host, const FmOutputs* out_host, int32_t lane, int32_t num_lanes, void* stream);
int fm_host_lane_range(const FmHandle* h, int32_t lane, int32_t num_lanes, int32_t* env_begin, int32_t* env_end);
int fm_reset_host(FmHandle* h, const uint8_t* mask_host, const FmOutputs* out_host, void* stream);
/* Info rows of the most recent fm_step_host call, copied to host on demand ([B, N, 14] floats).
 * The runner reads infos only at log time (graph_mpe_runner.py:143-146), so fm_step_host does not
 * copy them unless out_host->info is set. */
int fm_read_info_host(FmHandle* h, float* info_host, void* stream);

/* State injection / extraction (the reference has no API for this; tests assign
 * entity.state.* and world.* directly -- SURVEY.md section 8c). */
int fm_set_state(FmHandle* h, const FmState* st, void* stream);
int fm_get_state(FmHandle* h, const FmState* st, void* stream);

/* marl_fair_assign.solve_fair_assignment (marl_fair_assign.py:16-55), batched: one problem per
 * lane group.  costs: double [num, n, n] (cost[i][j] = agent i -> goal j); out: int32 [num, n]
 * goal index per agent (np.where(x == 1)[1], navigation_graph.py:558).  n <= 32.  Entries are
 * totally ordered by (cost, i, j), so tied costs have exactly one answer (oracle/lexifair.py).  A
 * problem with any NaN or +-inf cost gets -1 in every entry of its row; the other problems of the
 * batch are unaffected.  num == 0 does nothing (the pointers may be NULL). */
int fm_assign_costs(int device, const double* costs, int32_t num, int32_t n, int32_t* out, void* stream);
/* Same from positions: cdist(agent_pos, goal_pos) (navigation_graph.py:555) in float64 from
 * float [num, n, 2] inputs; a NaN or +-inf coordinate makes its problem's row -1. */
int fm_assign_positions(int device, const float* agent_pos, const float* goal_pos, int32_t num,
                        int32_t n, int32_t* out, void* stream);

/* scipy.optimize.linear_sum_assignment (nav_base_formation_graph_mask.py:255-260), batched, square problems, minimise:
 * one problem per warp, scipy's shortest augmenting path with its operation order and tie rule.  costs: double
 * [num, n, n]; out: int32 [num, n], out[p][i] = goal of agent i in problem p, equal to scipy's col_ind bit for bit (ties
 * included).  n <= 32.  A problem with any NaN or +-inf cost gets -1 in every entry of its row (scipy raises or reports
 * it infeasible); the other problems of the batch are unaffected.  num == 0 does nothing (the pointers may be NULL). */
int fm_assign_min_sum_costs(int device, const double* costs, int32_t num, int32_t n, int32_t* out, void* stream);
/* Same from positions: costs = float64 Euclidean distances of float [num, n, 2] inputs, as fm_assign_positions; a NaN or
 * +-inf coordinate makes its problem's row -1. */
int fm_assign_min_sum_positions(int device, const float* agent_pos, const float* goal_pos, int32_t num, int32_t n,
                                int32_t* out, void* stream);

/* Float64 Euclidean distances of `num` pairs of float [.,2] points, out[k] = ||a[k] - b[k]||: the kernels'
 * distance primitive (np.linalg.norm in World.calculate_distances, core.py:204-228; cdist at
 * navigation_graph.py:555), exposed so that its bit-exactness against numpy can be tested directly. */
int fm_pair_dist(int device, const float* a, const float* b, int64_t num, double* out, void* stream);

/* Policy-side edge list, TransformerConvNet.process_adj (onpolicy/algorithms/utils/gnn_new.py:381-413)
 * on adj float [num_graphs, E, E]: mask (adj < max_edge_dist) & (adj > 0) (inclusive != 0: <=, the
 * env-side Scenario.update_graph rule, navigation_graph.py:1037-1056), edges in (b, i, j) order.
 * repeat >= 1 emits every graph `repeat` times consecutively (graph b*repeat + a, node offset
 * (b*repeat + a)*E): the [B*N, E, E] batch the policy sees repeats each env's adj N times.
 * graph_offsets: int64 [num_graphs*repeat + 1] exclusive prefix of edge counts (out);
 * edge_index: int64 [2, capacity]; edge_attr: float [capacity]; nnz_out: int64 [1] (device, may be NULL).
 * Edges beyond `capacity` are not written, nnz_out still counts them (capacity num_graphs*repeat*E*E always suffices;
 * num_graphs*repeat*E*(E-1) for distance matrices, whose diagonal is zero). */
int fm_edge_list(int device, const float* adj, int32_t num_graphs, int32_t E, double max_edge_dist,
                 int32_t inclusive, int32_t repeat, int64_t capacity, int64_t* graph_offsets,
                 int64_t* edge_index, float* edge_attr, int64_t* nnz_out, void* stream);

/* Episode statistics (what base_runner.process_infos aggregates, base_runner.py:197-276).
 * Layout of the vector, K = fm_stats_len(N) doubles:
 *   [0 .. N)            sum of rewards per agent over all env-steps since the last clear
 *   [N .. N + 14 N)     per agent, the 14 info values summed over envs at their terminal step
 *   [15 N]              finished episodes,   [15 N + 1]  env-steps
 * fm_stats_read reduces the per-warp partial sums in a fixed order (deterministic) into
 * out_dev (device, K doubles); the caller all-reduces it across ranks (NCCL sum).  The formation family has the same
 * vector through fm_formation_stats_enable / fm_formation_stats_read (below). */
int fm_stats_len(int32_t num_agents);
int fm_stats_read(FmHandle* h, double* out_dev, int32_t clear, void* stream);

/* Introspection. */
int fm_num_entities(const FmHandle* h);
int fm_mapping(const FmHandle* h);                        /* 1 group-per-env, 2 agent-warp */
int64_t fm_algorithmic_bytes_per_step(const FmHandle* h); /* SURVEY.md section 8(d): W * 4 * B */
int fm_kernel_launches(const FmHandle* h, int64_t* out);   /* kernels launched by this handle so far */
int fm_abi_version(void);
const char* fm_last_error(void);

/* ---------------------------------------------------------------------------------------------------------------
 * Formation-family scenarios (SURVEY.md section 8f, N3): nav_fairassign_fairrew_formation_graph.py (fairness_reward 1)
 * and nav_fairassign_nofairrew_formation_graph.py (0) -- and, through `assignment`, the base scenarios of model_weights/OA
 * and RA -- under MultiAgentGraphEnv.step (environment.py:816-877).  Own handle; num_agents 2..7, 0..2 walls, relative node
 * features.  The sequential per-agent logic runs one thread per env; the outputs are emitted warp-cooperatively through
 * shared-memory images and TMA bulk stores (csrc/fm_formation.cu).  Outputs use FmOutputs with obs [B, N, 11] (:840-1015), node_obs [B, N, E, 13] (:1222-1340), adj [B, E, E],
 * reward / done [B, N], info [B, N, 14] (terminal values survive the auto-reset). */
#define FM_FORMATION_OBS_DIM 11
#define FM_FORMATION_NODE_FEAT_DIM 13
#define FM_FORMATION_MAX_OBSTACLES 8

typedef struct FmFormationConfig {
  int32_t num_envs, num_agents, num_obstacles, episode_length;
  int64_t env_offset;      /* global index of env 0 (Philox stream key; sharding does not change results) */
  uint64_t seed;
  double world_size, max_speed /* <= 0: None */, collision_rew, goal_rew, min_dist_thresh;
  double min_obs_dist;     /* onpolicy/config.py:188 */
  double fair_rew, zeroshift;
  int32_t fairness_reward; /* 1: ..._fairrew_... (tanh fairness term, :770-786); 0: ..._nofairrew_... */
  int32_t collaborative;   /* environment.py:867-870 */
  int32_t auto_reset;      /* graphworker, env_wrappers.py:859-865: reset once ALL agents of an env are done */
  int32_t assignment;      /* which goal an agent is rewarded for: 0 'fair' lexifair re-solved every step (:704-721; FA+FR, FA);
                              1 'optimal' min-sum matching re-solved every step (nav_base_formation_graph_mask.py:666-706; OA),
                              equal to scipy's linear_sum_assignment; 2 'random' permutation drawn at reset (nav_base_formation_graph_randomgoal.py:
                              258-259; RA).  1 and 2 use the base scenarios' 1.5x goal clearance and need fairness_reward 0. */
  int32_t info_every_step; /* 0: info rows are written on the steps on which every agent of the env is done (what the runner reads) */
  int32_t num_walls;       /* 0..2 (:301-333; core.py:36-55, :407-462): E = 2 N + O + W, wall rows of type 3 (:1323-1334) */
} FmFormationConfig;

/* State in API layout; the handle keeps it in exactly this layout (device), get / set are copies.  NULL: skipped. */
typedef struct FmFormationState {
  float* pos;                      /* [B, N, 2] */
  float* vel;                      /* [B, N, 2] */
  float* p_dist;                   /* [B, N] */
  float* landmark_pos;             /* [B, N, 2]  scenario.landmark_poses */
  float* obstacle_pos;             /* [B, O, 2] */
  int32_t* goal_match;             /* [B, N]  re-solved every step (:704-721) */
  float* dists_to_goal;            /* [B, N] */
  float* times_required;           /* [B, N] */
  float* dist_left_to_goal;        /* [B, N] */
  float* num_agent_collisions;     /* [B, N] */
  float* num_obstacle_collisions;  /* [B, N] */
  float* dist_traveled_mean;       /* [B] */
  float* dist_traveled_stddev;     /* [B] */
  int32_t* step;                   /* [B] */
  float* min_time;                 /* [B, N] */
  int32_t* episode;                /* [B] */
  uint8_t* status;                 /* [B, N]  agent.status (:408, :728; core.py:397-398; environment.py:240-242) */
  float* goal_reached;             /* [B, N]  scenario.goal_reached, -1 = none */
  float* occupied;                 /* [B, N]  scenario.landmark_poses_occupied */
  float* goal_history;             /* [B, N]  scenario.goal_history, -1 = none */
  float* wall_axis;                /* [B, W]  wall.axis_pos (:301-304) */
  int32_t* wall_orient;            /* [B, W]  0 'H', 1 'V' (:306) */
  float* wall_len;                 /* [B]     half-length, redrawn at every reset (:233-234) */
} FmFormationState;

typedef struct FmFormation FmFormation;

int fm_formation_create(const FmFormationConfig* cfg, int device, FmFormation** out);
int fm_formation_destroy(FmFormation* h);
/* env.reset() (environment.py:882-898 over reset_world / random_scenario, :217-487): mask uint8 [B] or NULL (= all);
 * every env is (re-)observed into `out` -- which, as in the reference, updates the goal-occupancy table. */
int fm_formation_reset(FmFormation* h, const uint8_t* mask, const FmOutputs* out, void* stream);
/* actions: int32 [B, N] in {0..4} (0 no-op, 1 +x, 2 -x, 3 +y, 4 -y). */
int fm_formation_step(FmFormation* h, const int32_t* actions, const FmOutputs* out, void* stream);
/* T consecutive steps with pre-generated actions int32 [T, B, N] (random-action rollouts, replayed trajectories): step t
 * writes outs[t] (host array of T FmOutputs of device pointers): one call, no host work between the steps.  With
 * FM_FORM_LANES=2 the batch runs as two env-range lanes on two streams forked from / joined to `stream` (measured no faster
 * for this family, DESIGN.md section 9).  Bit-identical to T calls of fm_formation_step either way. */
int fm_formation_step_many(FmFormation* h, const int32_t* actions, int32_t T, const FmOutputs* outs, void* stream);
int fm_formation_set_state(FmFormation* h, const FmFormationState* st, void* stream);
int fm_formation_get_state(FmFormation* h, const FmFormationState* st, void* stream);
/* Episode statistics of the formation steps: the vector of fm_stats_read, same layout and meaning (K = fm_stats_len(N)).
 * Per agent the emitted reward (the team total when collaborative) over all env-steps; per agent the 14 info values over
 * the envs whose agents are all done on that step (once per episode with auto_reset); the number of such envs; env-steps.
 * Resets add nothing.  Off by default (the logic kernel is a latency-bound chain at its register cap): enable != 0
 * allocates and clears the per-warp partial sums on first use and attaches them to the steps that follow; 0 detaches them
 * (they keep their values).  While on, a step whose caller passes no info array writes the info rows into the handle's
 * own, so the sums do not depend on which outputs are requested.  fm_formation_stats_read reduces the partial sums in a
 * fixed order (deterministic) into out_dev (device, K doubles) and zeroes them if `clear`; it fails while statistics are
 * off. */
int fm_formation_stats_enable(FmFormation* h, int32_t enable, void* stream);
int fm_formation_stats_read(FmFormation* h, double* out_dev, int32_t clear, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Fused graph-network forward of the rollout policy (SURVEY.md section 8f, row N2).
 * Replaces GNNBase.forward (onpolicy/algorithms/utils/gnn_new.py:555-575): process_adj (:381-413) -> EmbedConv
 * (:23-141) -> act(TransformerConv) x conv_layers (:252-271) -> node gather / global pool, for `num_graphs` graphs of
 * `num_entities` nodes each, in one kernel launch.  Shape family: embed_hidden_size = gnn_hidden_size = 16,
 * gnn_num_heads = 3, gnn_concat_heads = False (every shipped model_weights config).
 *   weights   device, fm_gnn_weight_floats() floats, packed as (row-major, H = 16):
 *               Wn[16][H]   lin1 weight, node-feature part, transposed; rows >= node_feat_dim - 1 zero
 *               T[4][H]     lin1[:, emb part] . entity_embed[type] + lin1 bias
 *               wd[H]       lin1 weight column of the edge attribute
 *               ln1 gamma[H], beta[H]
 *               embed_layers x { Wh[H in][H out], b[H], gamma[H], beta[H] }
 *               conv_layers  x { W[H][160] = [query | key | value | skip] transposed, b[160], w_edge[48] }
 *   node_obs  device [num_graphs, E, node_feat_dim]  (last column: entity type)
 *   adj       device [num_graphs / graphs_per_adj, E, E]: graph m reads matrix m / graphs_per_adj
 *   agent_id  device int32 [num_graphs] node gathered when aggr == 0 (NULL: m % graphs_per_adj)
 *   out       device [num_graphs, 16]
 * Two kernel mappings compute it (fm_policy.cu): one WARP per graph (gnn_kernel<E, RELU>, compiled for the E values of
 * FM_GNN_CASES), and one CTA per graph (gnn_wide_kernel<EMAX, RELU>, EMAX 32 or 64) for any 2 <= E <= 64 known at run
 * time.  Both are fp32, deterministic and batch-invariant; they may differ from each other in the last bits.
 */
typedef struct FmGnnConfig {
  int32_t num_graphs, graphs_per_adj, num_entities, node_feat_dim;
  int32_t embed_layers;     /* embed_layer_N (hidden layers of EmbedConv after lin1), 0..2 */
  int32_t conv_layers;      /* 1 + gnn_layer_N */
  int32_t aggr;             /* 0 node gather, 1 global mean, 2 global max, 3 global add */
  int32_t relu;             /* 1 ReLU, 0 Tanh (embed_use_ReLU == gnn_use_ReLU) */
  int32_t layer_norm;       /* use_feature_normalization */
  int32_t mapping;          /* 0 auto (= fm_gnn_mapping), 1 warp per graph (FM_ERR_UNSUPPORTED where E is not compiled),
                               2 CTA per graph (any 2 <= E <= 64); anything else FM_ERR_INVALID_ARG */
  double max_edge_dist;
} FmGnnConfig;
int64_t fm_gnn_weight_floats(const FmGnnConfig* cfg);
/* 1 if the warp-per-graph kernel (mapping 1) is compiled for this graph size */
int fm_gnn_supported(int32_t num_entities, int32_t node_feat_dim);
/* the mapping that auto (0) selects for this graph size: 1 where the warp-per-graph kernel is compiled, else 2 for
 * 2 <= E <= 64; 0 when no fused kernel covers it (E < 2, E > 64, or node_feat_dim outside 2..17) */
int fm_gnn_mapping(int32_t num_entities, int32_t node_feat_dim);
int fm_gnn_forward(int device, const FmGnnConfig* cfg, const float* weights, const float* node_obs, const float* adj,
                   const int32_t* agent_id, float* out, void* stream);
/* The same forward with a multi-node gather as the epilogue (GNNBase with graph_aggr='node' and k node indices per graph,
 * e.g. GR_Critic with critic_graph_aggr='node' gathering the N agent nodes through share_agent_id): the final states of
 * the k nodes agent_id[m][0..k-1] side by side.  cfg as for fm_gnn_forward except that cfg->aggr must be 0;
 *   agent_id  device int32 [num_graphs, k], 1 <= k <= num_entities (required)
 *   out       device [num_graphs, k * 16];  out[m][16 i + c] = fm_gnn_forward's out for the one-node gather agent_id[m][i]
 * Same mappings and weights as fm_gnn_forward; its kernels are the same code up to the epilogue. */
int fm_gnn_gather(int device, const FmGnnConfig* cfg, int32_t k, const float* weights, const float* node_obs,
                  const float* adj, const int32_t* agent_id, float* out, void* stream);

/* Fused policy head behind the graph network: GR_Actor.forward / GR_Critic.forward after gnn_base
 * (onpolicy/algorithms/graph_actor_critic.py:150-178, :380-397): [obs | nbd] -> MLPBase (utils/mlp.py) -> one GRU step
 * on h * mask + LayerNorm (utils/rnn.py:23-28, :57) -> Categorical head (utils/act.py; log-softmax, mode or a draw by
 * inverse CDF from the caller's uniforms, log-prob of the action) or the value layer.  hidden_size = 64, recurrent_N = 1.
 *   weights  device, fm_head_weight_floats() floats (W^T stored k-quad interleaved: [k / 4][column][4]):
 *              feature_norm gamma[32], beta[32] (input width obs_dim + 16 <= 32, zero padded)
 *              fc1 [8][64][4], b[64], ln gamma[64], beta[64];   layers x { [16][64][4], b, gamma, beta }
 *              recurrent: W_ih [16][192][4], W_hh [16][192][4], b_ih[192], b_hh[192], ln gamma[64], beta[64]
 *              output W[8 rows][64] (rows >= num_outputs zero), b[8]
 *   obs [rows, obs_dim] (NULL when obs_dim == 0), nbd [rows, 16], rnn_in [rows, 64], mask [rows], u [rows] or NULL (mode)
 *   rnn_out [rows, 64];  actor (value == NULL): action int64 [rows], logp [rows];  critic: value [rows] */
typedef struct FmHeadConfig {
  int32_t num_rows, obs_dim;
  int32_t layers;           /* layer_N: hidden layers after fc1, 0..2 */
  int32_t recurrent;        /* use_recurrent_policy or use_naive_recurrent_policy */
  int32_t feature_norm;     /* use_feature_normalization (the input LayerNorm) */
  int32_t relu;             /* use_ReLU */
  int32_t num_outputs;      /* actions (<= 8) or 1 for the critic */
  int32_t reserved_;
} FmHeadConfig;
int64_t fm_head_weight_floats(const FmHeadConfig* cfg);
int fm_policy_head(int device, const FmHeadConfig* cfg, const float* weights, const float* obs, const float* nbd,
                   const float* rnn_in, const float* mask, const float* u, float* rnn_out, float* logp, int64_t* action,
                   float* value, void* stream);

/* Fused critic head for wide inputs: GR_Critic.forward after gnn_base (graph_actor_critic.py:323-397) on
 * x = [cent_obs | nbd] of D = cent_dim + nbd_dim features, 1 <= D <= 768: feature LayerNorm over all D inputs ->
 * MLPBase -> one GRU step on h * mask + LayerNorm -> v_out.  It covers use_cent_obs (cent_obs = share_obs: the N agents'
 * observations side by side, cent_dim = N * obs_dim) and critic_graph_aggr='node' (nbd = fm_gnn_gather's k = N node
 * states, nbd_dim = N * 16), where fm_policy_head (obs_dim + 16 <= 32) does not.  hidden_size = 64, recurrent_N = 1.
 *   weights  device, fm_critic_head_weight_floats() floats; Dp = D rounded up to a multiple of 32 (zero padded):
 *              feature_norm gamma[Dp], beta[Dp]
 *              fc1 [Dp / 4][64][4] (W^T k-quad interleaved), b[64], ln gamma[64], beta[64]
 *              then exactly fm_policy_head's blob after its fc1 block: layers x { [16][64][4], b, gamma, beta },
 *              recurrent: W_ih [16][192][4], W_hh [16][192][4], b_ih[192], b_hh[192], ln gamma[64], beta[64],
 *              output W[8 rows][64] (row 0 = v_out, the rest zero), b[8]
 *   cent_obs [num_rows / rows_per_env, cent_dim]: ONE row per env, read by its rows_per_env consecutive rows (NULL when
 *            cent_dim == 0; num_rows must be a multiple of rows_per_env)
 *   nbd [rows, nbd_dim], rnn_in [rows, 64], mask [rows] (recurrent), rnn_out [rows, 64] (recurrent), value [rows]
 * fp32 on CUDA cores, deterministic and batch-invariant (the bits of a row do not depend on the batch around it). */
typedef struct FmCriticHeadConfig {
  int32_t num_rows;
  int32_t cent_dim;         /* N * obs_dim with use_cent_obs, else 0 */
  int32_t rows_per_env;     /* rows that share one cent_obs row (N) */
  int32_t nbd_dim;          /* 16 (global pool) or k * 16 (fm_gnn_gather) */
  int32_t layers;           /* layer_N: hidden layers after fc1, 0..2 */
  int32_t recurrent;        /* use_recurrent_policy or use_naive_recurrent_policy */
  int32_t feature_norm;     /* use_feature_normalization (the input LayerNorm) */
  int32_t relu;             /* use_ReLU */
} FmCriticHeadConfig;
int64_t fm_critic_head_weight_floats(const FmCriticHeadConfig* cfg);
int fm_critic_head(int device, const FmCriticHeadConfig* cfg, const float* weights, const float* cent_obs, const float* nbd,
                   const float* rnn_in, const float* mask, float* rnn_out, float* value, void* stream);

/* Training side of the device rollout buffer (fm_buffer.cu; fair-marl_b200/rollout.py DeviceRolloutBuffer): what
 * GraphReplayBuffer.compute_returns, the advantage lines of GR_MAPPO.train and the buffer's three mini-batch generators
 * compute (onpolicy/utils/graph_buffer.py, onpolicy/algorithms/graph_mappo.py).  Every field is a dense float32 array in
 * the buffer's layout: slab t of a [T(+1), B, N] field starts at t * B * N.  fp32 on CUDA cores with each operation rounded
 * on its own in the reference's order, deterministic, no atomics, no host synchronisation (graph-capturable).
 * A value normaliser (ValueNorm / PopArt) enters as two device floats, norm_mean and norm_std = sqrt(var), which its
 * denormalize applies as x * std + mean; both NULL means none.
 * Refusals (FM_ERR_INVALID_ARG, before the device is touched): a null required pointer, a dimension < 1, T * B * N >= 2^31. */
typedef struct FmReturnsConfig {
  int32_t episode_length, num_envs, num_agents;
  int32_t use_gae;
  int32_t use_proper_time_limits;
  int32_t reserved_;
  float gamma;              /* float(gamma) */
  float gamma_lambda;       /* float(gamma * gae_lambda), the product taken in double */
} FmReturnsConfig;
/* next_value [B, N] is stored into value_preds[T] (use_gae) or returns[T] (not), as the reference does, then for t =
 * T-1 .. 0 returns[t] follows every branch of compute_returns.  value_preds, returns, masks, bad_masks: [T+1, B, N];
 * rewards [T, B, N]; bad_masks is read only with use_proper_time_limits (may be NULL otherwise). */
int fm_buffer_returns(int device, const FmReturnsConfig* cfg, const float* next_value, float* value_preds, const float* rewards,
                      const float* masks, const float* bad_masks, const float* norm_mean, const float* norm_std,
                      float* returns, void* stream);

/* advantages[:T] = returns[:T] - denormalize(value_preds[:T]), then (adv - mean) / (std + 1e-5) with mean and the
 * population std (ddof 0) of the entries whose active_masks[:T] != 0, accumulated in fp64 (Welford / Chan, fixed order)
 * and rounded to float32; with no active entry both are NaN, as numpy's nanmean / nanstd give.
 *   stats      device float[2]: mean, std as used
 *   workspace  device double[FM_ADV_WORKSPACE_DOUBLES] (scratch; two launches) */
#define FM_ADV_WORKSPACE_DOUBLES 768
int fm_buffer_advantages(int device, int32_t episode_length, int32_t num_envs, int32_t num_agents, const float* returns,
                         const float* value_preds, const float* active_masks, const float* norm_mean, const float* norm_std,
                         float* advantages, float* stats, double* workspace, void* stream);

/* One mini-batch of an epoch of GraphReplayBuffer.feed_forward_generator / recurrent_generator /
 * naive_recurrent_generator in one launch, given the epoch's permutation (int64, as torch.randperm draws it):
 *   feed-forward  samples i = (t B + b) N + n, perm over T B N; per = mini_batch_size or T B N / num_mini_batch;
 *                 row j reads sample perm[k per + j]; rnn states of each row's own sample (per rows)
 *   recurrent     f = (b N + n) T + t, chunks = T B N / L, per = chunks / num_mini_batch, perm over the chunks; row
 *                 l per + c reads f = perm[k per + c] L + l (a chunk runs on into the next column when T % L != 0, as in
 *                 the reference); rnn states at each chunk's first step (per rows)
 *   naive         columns j = b N + n, per = B N / num_mini_batch (B N must divide), perm over B N; row t per + c reads
 *                 column perm[k per + c] at time t; rnn states at t = 0 (per rows)
 * share_obs is read from the env's obs row, adj from adj_env[t, b], agent_id / share_agent_id are synthesised from n.
 * Refusals besides the common ones: mode outside 0..2, data_chunk_length < 1 (recurrent), num_mini_batch < 1 or more
 * mini-batches than samples / chunks / columns, num_mini_batch * mini_batch_size > T B N, B N not divisible by
 * num_mini_batch (naive: the reference would then yield another number of mini-batches, or raise IndexError part-way
 * through the epoch), mini_batch outside 0..num_mini_batch-1. */
enum { FM_MINIBATCH_FEED_FORWARD = 0, FM_MINIBATCH_RECURRENT = 1, FM_MINIBATCH_NAIVE_RECURRENT = 2 };
typedef struct FmMinibatchConfig {
  int32_t episode_length, num_envs, num_agents, num_entities;
  int32_t obs_dim, node_feat_dim;
  int32_t rnn_floats;       /* recurrent_N * hidden_size */
  int32_t mode;             /* FM_MINIBATCH_* */
  int32_t num_mini_batch;
  int32_t mini_batch_size;  /* feed-forward: samples per mini-batch, 0 = T B N / num_mini_batch; must be 0 otherwise */
  int32_t data_chunk_length;
  int32_t mini_batch;       /* k: which mini-batch of the epoch */
} FmMinibatchConfig;
typedef struct FmBufferSlabs {         /* device pointers, all required */
  const float* obs;                    /* [T+1, B, N, obs_dim] */
  const float* node_obs;               /* [T+1, B, N, E, node_feat_dim] */
  const float* adj_env;                /* [T+1, B, E, E] */
  const float* rnn_states;             /* [T+1, B, N, rnn_floats] */
  const float* rnn_states_critic;
  const float* actions;                /* [T, B, N] */
  const float* action_log_probs;       /* [T, B, N] */
  const float* value_preds;            /* [T+1, B, N] */
  const float* returns;
  const float* masks;
  const float* active_masks;
  const float* advantages;             /* [T, B, N] */
} FmBufferSlabs;
typedef struct FmMinibatch {           /* device pointers, all required; R rows, R' = per rnn-state rows */
  float* share_obs;                    /* [R, N * obs_dim] */
  float* obs;                          /* [R, obs_dim] */
  float* node_obs;                     /* [R, E, node_feat_dim] */
  float* adj;                          /* [R, E, E] */
  int32_t* agent_id;                   /* [R] */
  int32_t* share_agent_id;             /* [R, N] */
  float* rnn_states;                   /* [R', rnn_floats] */
  float* rnn_states_critic;
  float* actions;                      /* [R] each */
  float* value_preds;
  float* returns;
  float* masks;
  float* active_masks;
  float* old_action_log_probs;
  float* adv_targ;
} FmMinibatch;
int fm_buffer_minibatch(int device, const FmMinibatchConfig* cfg, const FmBufferSlabs* in, const int64_t* perm,
                        const FmMinibatch* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FAIRMARL_H_ */
