// Host-callable launchers implemented in fm_kernels.cu (internal to libfairmarl.so).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "../../include/fairmarl.h"

namespace fm {
struct DevParams;
typedef FmState HostState;   // API-layout device pointers

int group_size(int n);
int num_warps(int B, int N);
// agent-warp mapping (fm_aw.cu): compiled for a fixed list of small (N, O)
bool aw_supported(int N, int O, int W = 0);
int aw_stats_rows(int B);
cudaError_t aw_prepare(const DevParams& p);
cudaError_t aw_launch(const DevParams& p, cudaStream_t st, bool is_reset);
// persistent rollout kernel of the agent-warp mapping (fm_roll.cu): num_steps <= FM_ROLL_MAX_STEPS env steps in one launch
#define FM_ROLL_MAX_STEPS 32
struct RollLaunch {
  int num_steps;
  int early;                 // every step writes its own output arrays: a tile is released right after its state write-back
  int max_ctas;              // one wave: SMs x resident CTAs per SM
  int stagger_ns;            // start-up delay per CTA slot of an SM (0: none)
  void* ctl;                 // device control block (roll_ctl_bytes), zero between launches
  const int* act_idx;        // step t reads act_idx + t * act_stride, or act_onehot + t * act_stride
  const float* act_onehot;
  long long act_stride;      // elements between consecutive steps' actions
  const FmOutputs* outs;     // [num_steps] (host memory; copied into the kernel parameters)
};
size_t roll_ctl_bytes(int B);
cudaError_t roll_prepare(const DevParams& p, int* ctas_per_sm);
cudaError_t roll_launch(const DevParams& p, const RollLaunch& r, cudaStream_t st);
cudaError_t launch_static_dists(const DevParams& p, cudaStream_t st);   // recompute p.sdist from the static positions
cudaError_t prepare_kernels(const DevParams& p);   // opt in to > 48 KB dynamic shared memory, once per handle
cudaError_t launch_step(const DevParams& p, cudaStream_t st, bool is_reset);
cudaError_t launch_prefetch(const DevParams& p, cudaStream_t st);   // next-episode placement + assignment (group mapping)
cudaError_t launch_assign(const double* costs, const float* apos, const float* gpos, int num, int n, int* out,
                          cudaStream_t st);
// batched min-sum assignment, scipy linear_sum_assignment bit for bit (fm_lsap.cu): one warp per problem, n <= 32
cudaError_t launch_lsap(const double* costs, const float* apos, const float* gpos, int num, int n, int* out, cudaStream_t st);
cudaError_t launch_state_io(const DevParams& p, const HostState& hs, int to_internal, cudaStream_t st);
cudaError_t launch_state_init(const DevParams& p, cudaStream_t st);
cudaError_t launch_observe_soa(const DevParams& p, float* obs, float* node, float* adj, cudaStream_t st);   // fm_soa.cu
cudaError_t launch_finite_guard(const DevParams& p, int* flags, int* count, cudaStream_t st);
int edge_list_blocks(int num_graphs);             // CTAs of the edge-list kernels (8 graphs each): size of `blocksums`
cudaError_t launch_edge_list(const float* adj, int num_graphs, int E, float thr, int inclusive, int repeat,
                             long long capacity, int* counts, long long* blocksums, long long* graph_offsets,
                             long long* edge_index, float* edge_attr, long long* nnz_out, cudaStream_t st);
// streamed form (fm_edges.cu, the default): count / offsets / persistent emission
size_t edge_stream_scratch_bytes(int num_graphs);
cudaError_t launch_edge_list_stream(const float* adj, int num_graphs, int E, float thr, int inclusive, int repeat,
                                    long long capacity, void* scratch, long long* graph_offsets, long long* edge_index,
                                    float* edge_attr, long long* nnz_out, cudaStream_t st);
// single-pass form (fm_edges.cu)
size_t edge_fused_smem(int E);
size_t edge_fused_scratch_bytes(int num_graphs);
cudaError_t launch_edge_list_fused(const float* adj, int num_graphs, int E, float thr, int inclusive, int repeat,
                                   long long capacity, void* scratch, long long* graph_offsets, long long* edge_index,
                                   float* edge_attr, long long* nnz_out, cudaStream_t st);
cudaError_t launch_pair_dist(const float* a, const float* b, long long num, double* out, cudaStream_t st);
cudaError_t launch_stats_reduce(double* partial, int rows, int K, double* out, int clear, cudaStream_t st);

// formation family (fm_formation.cu): per-env logic one thread per env, warp-cooperative emission; state in API layout
struct FormParams {
  int B, N, O, episode_length, fairness_reward, collaborative, auto_reset, has_max_speed;
  int assignment;            // 0 fair (lexifair every step), 1 optimal (min-sum every step), 2 random (permutation at reset)
  int info_every_step;       // 0: info rows only on the steps on which every agent of the env is done
  long long env_offset;
  uint32_t seed_lo, seed_hi;
  double world_size, max_speed, collision_rew, goal_rew, min_dist_thresh, min_obs_dist, fair_rew, zeroshift;
  FmFormationState st;       // device pointers owned by the handle
  FmOutputs out;             // this launch
  const int32_t* actions;    // step
  const uint8_t* mask;       // reset
  float* rec;                // handle-owned recipe block of the split step path ([tiles][32][rec_stride] floats); null: fused kernel
  int fused;                 // 1: always the fused kernel (FM_FORM_FUSED=1, diagnostic / A-B)
  int W;                     // walls (0..2): fused generic kernel only; entities 2N+O .. E-1 are the wall midpoints
  float* pend;               // pending-reset blocks of the split step path ([form_pending_floats][Bp], fm_form.cuh); null: none
  int Bp;                    // B rounded up to whole warps
  int* ready;                // split step path: one flag per 16 envs, logic kernel -> image kernel (programmatic dependent launch); null: none
  double* stats;             // episode statistics, [ceil(B / 32)][15 N + 2] per-warp partial sums (fm_stats_read layout); null: off
};
size_t formation_recipe_floats(int N, int O, int B);
cudaError_t launch_formation_image(const FormParams& p, cudaStream_t st);   // fm_form_image.cu: node_obs / adj from p.rec
struct FormAsync { cudaStream_t side; cudaEvent_t fork, join; };   // handle-owned: the prefetch kernel runs beside the image kernel
size_t formation_pending_floats(int N, int O, int B);
cudaError_t launch_formation_prefetch(const FormParams& p, cudaStream_t st);   // fm_form_image.cu
cudaError_t launch_formation(const FormParams& p, bool is_reset, cudaStream_t st, const FormAsync* async = nullptr);
// fused graph-network forward of the rollout policy (fm_policy.cu)
bool gnn_supported_entities(int E);        // warp per graph (gnn_kernel<E, RELU>): compiled for E
constexpr int GNN_WIDE_MAX_ENTITIES = 2 * FM_MAX_AGENTS;
bool gnn_wide_supported_entities(int E);   // CTA per graph (gnn_wide_kernel<EMAX, RELU>): 2 <= E <= 64
int gnn_weight_count(int embed_layers, int conv_layers);
// gather_k 0: aggr as in FmGnnConfig (gnn_kernel / gnn_wide_kernel); gather_k >= 1: the final states of gather_k nodes per
// graph side by side (the GATHER instantiations, agent_id [M, gather_k])
cudaError_t launch_gnn(const FmGnnConfig& c, const float* weights, const float* node, const float* adj, const int* agent_id,
                       float* out, int gather_k, cudaStream_t st);
int head_weight_count(int layers, int recurrent);
cudaError_t launch_head(const FmHeadConfig& c, const float* weights, const float* obs, const float* nbd, const float* rnn_in,
                        const float* mask, const float* u, float* rnn_out, float* logp, long long* action, float* value,
                        cudaStream_t st);
constexpr int CRITIC_HEAD_MAX_IN = 768;    // critic_head_kernel: input width cap
int critic_head_weight_count(int in_dim, int layers, int recurrent);
cudaError_t launch_critic_head(const FmCriticHeadConfig& c, const float* weights, const float* cent_obs, const float* nbd,
                               const float* rnn_in, const float* mask, float* rnn_out, float* value, cudaStream_t st);
// training side of the rollout buffer (fm_buffer.cu); arguments checked by fm_abi.cu
cudaError_t launch_buffer_returns(const FmReturnsConfig& c, const float* next_value, float* value_preds, const float* rewards,
                                  const float* masks, const float* bad_masks, const float* norm_mean, const float* norm_std,
                                  float* returns, cudaStream_t st);
cudaError_t launch_buffer_advantages(long long n, const float* returns, const float* value_preds, const float* active_masks,
                                     const float* norm_mean, const float* norm_std, float* advantages, float* stats,
                                     double* workspace, cudaStream_t st);
// rows output rows, rnn_rows of them with rnn states, per samples / chunks / columns per mini-batch, off = k * per
cudaError_t launch_buffer_minibatch(const FmMinibatchConfig& c, long long rows, long long rnn_rows, int per, long long off,
                                    const FmBufferSlabs& in, const long long* perm, const FmMinibatch& out, cudaStream_t st);
int formation_max_agents();
int set_error(int code, const char* fmt, ...);   // fm_last_error text (fm_abi.cu)
}  // namespace fm
