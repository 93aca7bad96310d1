"""B200-native batched simulator for Fair-MARL's GraphMPE ``navigation_graph`` environment.

Host side: Python over a C ABI (``include/fairmarl.h``, ``libfairmarl.so``) of hand-written
sm_100a CUDA kernels.  There is no CPU path: every op raises if the library or a CUDA device is
missing.  Public surface mirrors the reference interfaces this package replaces:

* ``B200GraphVecEnv``  -- ``onpolicy/envs/env_wrappers.py`` ``GraphSubprocVecEnv`` (ShareVecEnv API)
* ``solve_fair_assignment`` / ``lexifair_batched`` -- ``marl_fair_assign.py``
* ``linear_sum_assignment`` / ``min_sum_batched`` -- ``scipy.optimize.linear_sum_assignment`` (square, minimise)
* ``process_adj`` -- ``onpolicy/algorithms/utils/gnn_new.py:381-413``
* ``DeviceRolloutBuffer`` / ``RolloutCollector`` -- ``onpolicy/utils/graph_buffer.py`` ``GraphReplayBuffer`` and the
  collect / insert loop of ``onpolicy/runner/shared/graph_mpe_runner.py`` (device-resident, written by the step kernel)
* ``B200FormationVecEnv`` -- the formation-family scenarios (``nav_fairassign_{fairrew,nofairrew}_formation_graph``), a first
  tensor-native device path (N <= 4)
* ``DenseGraphActor`` / ``DenseGraphCritic`` -- the forward pass of ``GR_Actor`` / ``GR_Critic`` without torch_geometric
"""
from fair_marl_b200.build import build_library, library_path            # noqa: F401
from fair_marl_b200.config import SimConfig                             # noqa: F401
from fair_marl_b200.spaces import Box, Discrete                         # noqa: F401
from fair_marl_b200.vec_env import B200GraphVecEnv, make_train_env      # noqa: F401
from fair_marl_b200.assign import (lexifair_batched, linear_sum_assignment, min_sum_batched, pair_dist,  # noqa: F401
                                    solve_fair_assignment)
from fair_marl_b200.edges import process_adj                            # noqa: F401
from fair_marl_b200.sharding import shard_range, EpisodeStats           # noqa: F401
from fair_marl_b200.policy import DenseGraphActor, DenseGraphCritic, PolicyConfig, load_reference_state_dict  # noqa: F401
from fair_marl_b200.rollout import DeviceRolloutBuffer, RolloutCollector  # noqa: F401
from fair_marl_b200.formation import B200FormationVecEnv, FormationSimConfig  # noqa: F401

__all__ = ["B200GraphVecEnv", "make_train_env", "SimConfig", "Box", "Discrete", "solve_fair_assignment",
           "lexifair_batched", "min_sum_batched", "linear_sum_assignment", "pair_dist", "process_adj", "shard_range", "EpisodeStats", "build_library", "library_path",
           "DenseGraphActor", "DenseGraphCritic", "PolicyConfig", "load_reference_state_dict", "DeviceRolloutBuffer",
           "RolloutCollector", "B200FormationVecEnv", "FormationSimConfig"]
