"""ctypes binding of ``libfairmarl.so`` (include/fairmarl.h).  Loading fails loudly: there is no
fallback implementation."""
from __future__ import annotations

import ctypes as C
import os

from fair_marl_b200.build import library_path

OBS_DIM, NODE_FEAT_DIM, INFO_DIM = 7, 11, 14
NODE_FEAT_DIM_GLOBAL = 7        # graph_feat_type = 'global'
INFO_KEYS = (
    "individual_reward", "Dist_to_goal", "Time_req_to_goal", "Num_agent_collisions",
    "Num_obst_collisions", "Distance_mean", "Distance_variance", "Mean_by_variance",
    "Dists_traveled", "Time_taken", "Time_mean", "Time_stddev", "Time_mean_by_stddev",
    "Min_time_to_goal",
)


class FmConfig(C.Structure):
    _fields_ = [
        ("num_envs", C.c_int32), ("num_agents", C.c_int32), ("num_obstacles", C.c_int32),
        ("episode_length", C.c_int32), ("env_offset", C.c_int64), ("seed", C.c_uint64),
        ("world_size", C.c_double), ("max_speed", C.c_double), ("collision_rew", C.c_double),
        ("goal_rew", C.c_double), ("min_dist_thresh", C.c_double), ("fair_rew", C.c_double),
        ("zeroshift", C.c_double), ("max_edge_dist", C.c_double),
        ("fairness_reward", C.c_int32), ("collaborative", C.c_int32), ("auto_reset", C.c_int32),
        ("info_every_step", C.c_int32), ("mapping", C.c_int32), ("graph_feat_global", C.c_int32),
        ("num_walls", C.c_int32), ("reserved_", C.c_int32),
    ]


class FmOutputs(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("node_obs", C.c_void_p), ("adj", C.c_void_p),
                ("reward", C.c_void_p), ("done", C.c_void_p), ("info", C.c_void_p)]


STATE_FIELDS = ("pos", "vel", "p_dist", "landmark_pos", "obstacle_pos", "goal_match", "dists_to_goal",
                "times_required", "dist_left_to_goal", "num_agent_collisions", "num_obstacle_collisions",
                "dist_traveled_mean", "dist_traveled_stddev", "step", "min_time", "episode",
                "wall_axis", "wall_orient", "wall_len")
STATE_INT_FIELDS = ("goal_match", "num_agent_collisions", "num_obstacle_collisions", "step", "episode", "wall_orient")


class FmSoaOutputs(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("node_obs", C.c_void_p), ("adj", C.c_void_p)]


class FmState(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in STATE_FIELDS]


# formation family (include/fairmarl.h: FmFormationConfig / FmFormationState)
FORMATION_OBS_DIM, FORMATION_NODE_FEAT_DIM, FORMATION_MAX_OBSTACLES = 11, 13, 8


class FmFormationConfig(C.Structure):
    _fields_ = [
        ("num_envs", C.c_int32), ("num_agents", C.c_int32), ("num_obstacles", C.c_int32), ("episode_length", C.c_int32),
        ("env_offset", C.c_int64), ("seed", C.c_uint64),
        ("world_size", C.c_double), ("max_speed", C.c_double), ("collision_rew", C.c_double), ("goal_rew", C.c_double),
        ("min_dist_thresh", C.c_double), ("min_obs_dist", C.c_double), ("fair_rew", C.c_double), ("zeroshift", C.c_double),
        ("fairness_reward", C.c_int32), ("collaborative", C.c_int32), ("auto_reset", C.c_int32), ("assignment", C.c_int32),
        ("info_every_step", C.c_int32), ("num_walls", C.c_int32),
    ]


FORMATION_STATE_FIELDS = ("pos", "vel", "p_dist", "landmark_pos", "obstacle_pos", "goal_match", "dists_to_goal",
                          "times_required", "dist_left_to_goal", "num_agent_collisions", "num_obstacle_collisions",
                          "dist_traveled_mean", "dist_traveled_stddev", "step", "min_time", "episode", "status",
                          "goal_reached", "occupied", "goal_history", "wall_axis", "wall_orient", "wall_len")
FORMATION_STATE_INT_FIELDS = ("goal_match", "step", "episode", "wall_orient")


class FmFormationState(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in FORMATION_STATE_FIELDS]


class FmGnnConfig(C.Structure):
    _fields_ = [("num_graphs", C.c_int32), ("graphs_per_adj", C.c_int32), ("num_entities", C.c_int32),
                ("node_feat_dim", C.c_int32), ("embed_layers", C.c_int32), ("conv_layers", C.c_int32), ("aggr", C.c_int32),
                ("relu", C.c_int32), ("layer_norm", C.c_int32), ("mapping", C.c_int32), ("max_edge_dist", C.c_double)]


class FmHeadConfig(C.Structure):
    _fields_ = [("num_rows", C.c_int32), ("obs_dim", C.c_int32), ("layers", C.c_int32), ("recurrent", C.c_int32),
                ("feature_norm", C.c_int32), ("relu", C.c_int32), ("num_outputs", C.c_int32), ("reserved_", C.c_int32)]


class FmCriticHeadConfig(C.Structure):
    _fields_ = [("num_rows", C.c_int32), ("cent_dim", C.c_int32), ("rows_per_env", C.c_int32), ("nbd_dim", C.c_int32),
                ("layers", C.c_int32), ("recurrent", C.c_int32), ("feature_norm", C.c_int32), ("relu", C.c_int32)]


class FmReturnsConfig(C.Structure):
    _fields_ = [("episode_length", C.c_int32), ("num_envs", C.c_int32), ("num_agents", C.c_int32), ("use_gae", C.c_int32),
                ("use_proper_time_limits", C.c_int32), ("reserved_", C.c_int32), ("gamma", C.c_float), ("gamma_lambda", C.c_float)]


MINIBATCH_MODES = {"feed_forward": 0, "recurrent": 1, "naive_recurrent": 2}     # FM_MINIBATCH_*
ADV_WORKSPACE_DOUBLES = 768                                                     # FM_ADV_WORKSPACE_DOUBLES


class FmMinibatchConfig(C.Structure):
    _fields_ = [(name, C.c_int32) for name in (
        "episode_length", "num_envs", "num_agents", "num_entities", "obs_dim", "node_feat_dim", "rnn_floats", "mode",
        "num_mini_batch", "mini_batch_size", "data_chunk_length", "mini_batch")]


BUFFER_SLAB_FIELDS = ("obs", "node_obs", "adj_env", "rnn_states", "rnn_states_critic", "actions", "action_log_probs",
                      "value_preds", "returns", "masks", "active_masks", "advantages")
MINIBATCH_FIELDS = ("share_obs", "obs", "node_obs", "adj", "agent_id", "share_agent_id", "rnn_states", "rnn_states_critic",
                    "actions", "value_preds", "returns", "masks", "active_masks", "old_action_log_probs", "adv_targ")


class FmBufferSlabs(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in BUFFER_SLAB_FIELDS]


class FmMinibatch(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in MINIBATCH_FIELDS]


class FairMarlError(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.isfile(path):
        raise FairMarlError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  fair_marl_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    sig = {
        "fm_abi_version": ([], C.c_int),
        "fm_last_error": ([], C.c_char_p),
        "fm_stats_len": ([i32], C.c_int),
        "fm_create": ([C.POINTER(FmConfig), C.c_int, C.POINTER(vp)], C.c_int),
        "fm_destroy": ([vp], C.c_int),
        "fm_reset": ([vp, vp, C.POINTER(FmOutputs), vp], C.c_int),
        "fm_observe": ([vp, C.POINTER(FmOutputs), vp], C.c_int),
        "fm_soa_stride": ([vp], C.c_int),
        "fm_observe_soa": ([vp, C.POINTER(FmSoaOutputs), vp], C.c_int),
        "fm_check_finite": ([vp, vp, vp, vp], C.c_int),
        "fm_step": ([vp, vp, C.POINTER(FmOutputs), vp], C.c_int),
        "fm_step_onehot": ([vp, vp, C.POINTER(FmOutputs), vp], C.c_int),
        "fm_step_many": ([vp, vp, i32, C.POINTER(FmOutputs), vp], C.c_int),
        "fm_step_host": ([vp, vp, C.POINTER(FmOutputs), vp], C.c_int),
        "fm_step_host_lane": ([vp, vp, C.POINTER(FmOutputs), i32, i32, vp], C.c_int),
        "fm_host_lane_range": ([vp, i32, i32, C.POINTER(i32), C.POINTER(i32)], C.c_int),
        "fm_reset_host": ([vp, vp, C.POINTER(FmOutputs), vp], C.c_int),
        "fm_read_info_host": ([vp, vp, vp], C.c_int),
        "fm_set_state": ([vp, C.POINTER(FmState), vp], C.c_int),
        "fm_get_state": ([vp, C.POINTER(FmState), vp], C.c_int),
        "fm_assign_costs": ([C.c_int, vp, i32, i32, vp, vp], C.c_int),
        "fm_assign_positions": ([C.c_int, vp, vp, i32, i32, vp, vp], C.c_int),
        "fm_assign_min_sum_costs": ([C.c_int, vp, i32, i32, vp, vp], C.c_int),
        "fm_assign_min_sum_positions": ([C.c_int, vp, vp, i32, i32, vp, vp], C.c_int),
        "fm_pair_dist": ([C.c_int, vp, vp, i64, vp, vp], C.c_int),
        "fm_edge_list": ([C.c_int, vp, i32, i32, C.c_double, i32, i32, i64, vp, vp, vp, vp, vp], C.c_int),
        "fm_stats_read": ([vp, vp, i32, vp], C.c_int),
        "fm_num_entities": ([vp], C.c_int),
        "fm_mapping": ([vp], C.c_int),
        "fm_algorithmic_bytes_per_step": ([vp], i64),
        "fm_kernel_launches": ([vp, C.POINTER(i64)], C.c_int),
        "fm_formation_create": ([C.POINTER(FmFormationConfig), C.c_int, C.POINTER(vp)], C.c_int),
        "fm_formation_destroy": ([vp], C.c_int),
        "fm_formation_reset": ([vp, vp, C.POINTER(FmOutputs), vp], C.c_int),
        "fm_formation_step": ([vp, vp, C.POINTER(FmOutputs), vp], C.c_int),
        "fm_formation_step_many": ([vp, vp, i32, C.POINTER(FmOutputs), vp], C.c_int),
        "fm_formation_set_state": ([vp, C.POINTER(FmFormationState), vp], C.c_int),
        "fm_formation_get_state": ([vp, C.POINTER(FmFormationState), vp], C.c_int),
        "fm_formation_stats_enable": ([vp, i32, vp], C.c_int),
        "fm_formation_stats_read": ([vp, vp, i32, vp], C.c_int),
        "fm_gnn_weight_floats": ([C.POINTER(FmGnnConfig)], i64),
        "fm_gnn_supported": ([i32, i32], C.c_int),
        "fm_gnn_mapping": ([i32, i32], C.c_int),
        "fm_gnn_forward": ([C.c_int, C.POINTER(FmGnnConfig), vp, vp, vp, vp, vp, vp], C.c_int),
        "fm_head_weight_floats": ([C.POINTER(FmHeadConfig)], i64),
        "fm_policy_head": ([C.c_int, C.POINTER(FmHeadConfig), vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp], C.c_int),
        "fm_gnn_gather": ([C.c_int, C.POINTER(FmGnnConfig), i32, vp, vp, vp, vp, vp, vp], C.c_int),
        "fm_critic_head_weight_floats": ([C.POINTER(FmCriticHeadConfig)], i64),
        "fm_critic_head": ([C.c_int, C.POINTER(FmCriticHeadConfig), vp, vp, vp, vp, vp, vp, vp, vp], C.c_int),
        "fm_buffer_returns": ([C.c_int, C.POINTER(FmReturnsConfig), vp, vp, vp, vp, vp, vp, vp, vp, vp], C.c_int),
        "fm_buffer_advantages": ([C.c_int, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp], C.c_int),
        "fm_buffer_minibatch": ([C.c_int, C.POINTER(FmMinibatchConfig), C.POINTER(FmBufferSlabs), vp, C.POINTER(FmMinibatch), vp],
                                C.c_int),
    }
    for name, (argtypes, restype) in sig.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export the ABI
        fn.argtypes, fn.restype = argtypes, restype
    _lib = lib
    return lib


EXPORTED_SYMBOLS = (
    "fm_abi_version", "fm_last_error", "fm_stats_len", "fm_create", "fm_destroy", "fm_reset", "fm_observe", "fm_soa_stride", "fm_observe_soa", "fm_check_finite", "fm_step",
    "fm_step_onehot", "fm_step_many", "fm_step_host", "fm_step_host_lane", "fm_host_lane_range", "fm_reset_host", "fm_read_info_host", "fm_set_state", "fm_get_state",
    "fm_assign_costs", "fm_assign_positions", "fm_assign_min_sum_costs", "fm_assign_min_sum_positions", "fm_pair_dist", "fm_edge_list", "fm_stats_read", "fm_num_entities", "fm_mapping",
    "fm_algorithmic_bytes_per_step", "fm_kernel_launches",
    "fm_formation_create", "fm_formation_destroy", "fm_formation_reset", "fm_formation_step", "fm_formation_step_many",
    "fm_formation_set_state",
    "fm_formation_get_state", "fm_formation_stats_enable", "fm_formation_stats_read", "fm_gnn_weight_floats", "fm_gnn_supported", "fm_gnn_mapping",
    "fm_gnn_forward",
    "fm_head_weight_floats", "fm_policy_head", "fm_gnn_gather", "fm_critic_head_weight_floats", "fm_critic_head",
    "fm_buffer_returns", "fm_buffer_advantages", "fm_buffer_minibatch",
)


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().fm_last_error().decode(errors="replace")
        raise FairMarlError(f"{what or 'libfairmarl'} failed ({rc}): {msg}")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise FairMarlError("no CUDA device visible: fair_marl_b200 has no CPU path")
    return torch
