"""Formation-family scenarios on the device -- ``nav_fairassign_fairrew_formation_graph`` (FA+FR), ``..._nofairrew_...``
(FA), ``nav_base_formation_graph_mask`` (OA) and ``nav_base_formation_graph_randomgoal`` (RA), i.e. the scenario files of the
four shipped ``model_weights`` -- as a tensor-native env over ``fm_formation_*`` (include/fairmarl.h; kernels in
csrc/fm_formation.cu: per-env logic one thread per env, warp-cooperative TMA emission; N = 2..7, 0..2 walls).

SURVEY.md section 8f, N3: device tensors in, device tensors out, the same dict keys
as ``B200GraphVecEnv.step_tensor`` with this family's shapes -- ``obs [B,N,11]`` (scenario ``observation``, :840-1015),
``node_obs [B,N,E,13]`` (``_get_entity_feat_relative``, :1222-1340), ``adj_env [B,E,E]``, ``reward [B,N]``,
``done [B,N]`` (per-agent early done, environment.py:240-242), ``info [B,N,14]``.  ``reset()`` / ``step()`` wrap the same
calls in the numpy tuples of ``GraphSubprocVecEnv`` (env_wrappers.py:983-1002) with the spaces the runner reads.
No CPU path: raises without the library or a CUDA device.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Any, Dict, Optional

import numpy as np

from fair_marl_b200 import _lib
from fair_marl_b200.spaces import Box, Discrete


# scenario file -> (assignment, fairness_reward): the four formation scenarios this path covers
SCENARIO_MODES = {"nav_fairassign_fairrew_formation_graph": ("fair", True), "nav_fairassign_nofairrew_formation_graph": ("fair", False),
                  "nav_base_formation_graph_mask": ("optimal", False), "nav_base_formation_graph_randomgoal": ("random", False)}


@dataclass
class FormationSimConfig:
    """The argparse fields the formation ``Scenario.make_world`` reads (:48-216) that this path honours."""
    num_agents: int = 3
    num_obstacles: int = 3
    world_size: float = 2.0
    max_speed: Optional[float] = 2.0
    collision_rew: float = 5.0
    goal_rew: float = 5.0
    min_dist_thresh: float = 0.05
    min_obs_dist: float = 0.5
    episode_length: int = 25
    fair_rew: float = 1.0
    zeroshift: float = 5.0
    collaborative: bool = False
    fairness_reward: bool = True       # True: ..._fairrew_... scenario; False: ..._nofairrew_...
    auto_reset: bool = True
    assignment: str = "fair"           # 'fair' (FA+FR, FA) | 'optimal' (OA: min-sum matching every step) | 'random' (RA)
    info_every_step: bool = True       # False: info rows only on the steps where every agent of the env is done (rollouts)
    num_walls: int = 0                 # 0..2 (:301-333): wall midpoints close the entity list, rows of type 3

    @property
    def num_entities(self) -> int:
        return 2 * self.num_agents + self.num_obstacles + self.num_walls

    @classmethod
    def from_args(cls, args: Any, **overrides) -> "FormationSimConfig":
        kw = {f: getattr(args, f) for f in cls.__dataclass_fields__ if hasattr(args, f)}
        name = getattr(args, "scenario_name", "nav_fairassign_fairrew_formation_graph")
        if name not in SCENARIO_MODES:
            raise NotImplementedError(f"scenario {name!r} is not one of the four formation scenarios this path covers")
        kw["assignment"], kw["fairness_reward"] = SCENARIO_MODES[name]
        for unsupported in ("num_scripted_agents",):
            if getattr(args, unsupported, 0):
                raise NotImplementedError(f"{unsupported} > 0 is not supported by the formation kernels")
        if getattr(args, "graph_feat_type", "relative") != "relative":
            raise NotImplementedError("the formation kernels emit the relative node features only")
        if hasattr(args, "num_landmarks") and args.num_landmarks != kw.get("num_agents", 3):
            raise ValueError("the formation scenarios need num_landmarks == num_agents")
        kw.update(overrides)
        return cls(**kw)


def decode_onehot_actions(actions_env, num_envs: int, num_agents: int) -> np.ndarray:
    """``[B,N,5]`` one-hot (graph_mpe_runner.py:429-431) or ``[B,N]`` indices -> int32 ``[B,N]``.  The reference decodes
    ``u = [a1 - a2, a3 - a4]`` (environment.py:301-311); for a one-hot row that is the move of its hot index, so anything
    that is not exactly one-hot is refused instead of being reinterpreted."""
    a = np.asarray(actions_env)
    if a.shape == (num_envs, num_agents):
        idx = a.astype(np.int64)
    elif a.shape == (num_envs, num_agents, 5):
        idx = a.argmax(axis=-1)
        if not (np.isin(a, (0, 1)).all() and (a.sum(axis=-1) == 1).all()):
            raise ValueError("actions must be exact one-hot rows over the 5 discrete moves")
    else:
        raise ValueError(f"actions must be [B,N,5] one-hot (or [B,N] indices), got {a.shape}")
    if idx.min(initial=0) < 0 or idx.max(initial=0) > 4:
        raise ValueError("action indices must be in 0..4")
    return idx.astype(np.int32)


def infos_from_rows(rows: np.ndarray, with_min_time: bool = True):
    """``[B,N,14]`` info rows -> the reference's ``infos``: B lists of N dicts (formation ``info_callback`` :538-575 +
    ``individual_reward``, environment.py:857)."""
    keys = _lib.INFO_KEYS if with_min_time else _lib.INFO_KEYS[:-1]
    return [[{k: float(rows[b, i, j]) for j, k in enumerate(keys)} for i in range(rows.shape[1])] for b in range(rows.shape[0])]


def share_vec_env_tuple(out: Dict[str, np.ndarray], with_min_time: bool = True):
    """numpy outputs of one step -> ``(obs, agent_id, node_obs, adj, rewards, dones, infos)`` as
    ``GraphSubprocVecEnv.step_wait`` stacks them (env_wrappers.py:988-996): ``adj`` per agent ``[B,N,E,E]`` (a broadcast
    view: the reference stores the same matrix N times), ``agent_id [B,N,1]`` = the agents' global ids 0..N-1 (:1017)."""
    obs = out["obs"]
    B, N = obs.shape[:2]
    E = out["adj_env"].shape[-1]
    agent_id = np.broadcast_to(np.arange(N, dtype=np.float32).reshape(1, N, 1), (B, N, 1))
    adj = np.broadcast_to(out["adj_env"][:, None], (B, N, E, E))
    head = (obs, agent_id, out["node_obs"], adj)
    if "reward" not in out:
        return head                                                    # reset(): the 4-tuple (env_wrappers.py:997-1002)
    return head + (out["reward"], out["done"].astype(bool), infos_from_rows(out["info"], with_min_time))


class B200FormationVecEnv:
    """B formation envs on one GPU.  ``reset_tensor()`` / ``step_tensor(actions int32 [B,N])`` return dicts of CUDA
    tensors (views of buffers owned by this object, overwritten by the next call), or of the caller's arrays with
    ``out=`` (e.g. the slabs of a ``DeviceRolloutBuffer``).  ``episode_stats``: the steps add up, on the device, the
    statistics vector of ``read_stats`` (off by default: it costs the step kernels a little)."""

    closed = False

    def __init__(self, cfg: FormationSimConfig, num_envs: int, device: int = 0, seed: int = 0, env_offset: int = 0,
                 num_slots: int = 1, episode_stats: bool = False):
        torch = _lib.require_cuda()
        self.torch, self.lib, self.cfg = torch, _lib.load(), cfg
        self.num_envs, self.num_agents, self.num_entities = int(num_envs), cfg.num_agents, cfg.num_entities
        self.device_index, self.device = int(device), torch.device("cuda", int(device))
        c = _lib.FmFormationConfig(
            num_envs=self.num_envs, num_agents=cfg.num_agents, num_obstacles=cfg.num_obstacles,
            episode_length=cfg.episode_length, env_offset=int(env_offset), seed=int(seed) & (2 ** 64 - 1),
            world_size=cfg.world_size, max_speed=cfg.max_speed if cfg.max_speed is not None else -1.0,
            collision_rew=cfg.collision_rew, goal_rew=cfg.goal_rew, min_dist_thresh=cfg.min_dist_thresh,
            min_obs_dist=cfg.min_obs_dist, fair_rew=cfg.fair_rew, zeroshift=cfg.zeroshift,
            fairness_reward=int(cfg.fairness_reward), collaborative=int(cfg.collaborative), auto_reset=int(cfg.auto_reset),
            assignment={"fair": 0, "optimal": 1, "random": 2}[cfg.assignment], info_every_step=int(cfg.info_every_step), num_walls=int(cfg.num_walls))
        self._h = C.c_void_p()
        _lib.check(self.lib.fm_formation_create(C.byref(c), self.device_index, C.byref(self._h)), "fm_formation_create")
        B, N, E = self.num_envs, self.num_agents, self.num_entities
        f32 = dict(dtype=torch.float32, device=self.device)
        # `num_slots` sets of output buffers, used round robin (1: every call overwrites the previous results)
        info = torch.zeros((B, N, _lib.INFO_DIM), **f32)
        self._slots = [{
            "obs": torch.zeros((B, N, _lib.FORMATION_OBS_DIM), **f32),
            "node_obs": torch.zeros((B, N, E, _lib.FORMATION_NODE_FEAT_DIM), **f32),
            "adj_env": torch.zeros((B, E, E), **f32), "reward": torch.zeros((B, N), **f32),
            "done": torch.zeros((B, N), dtype=torch.uint8, device=self.device),
            "info": info} for _ in range(max(1, int(num_slots)))]
        self._outs = [_lib.FmOutputs(b["obs"].data_ptr(), b["node_obs"].data_ptr(), b["adj_env"].data_ptr(),
                                     b["reward"].data_ptr(), b["done"].data_ptr(), b["info"].data_ptr()) for b in self._slots]
        self._slot = 0
        self._buf = self._slots[0]
        inf, No, Nn = float("inf"), _lib.FORMATION_OBS_DIM, _lib.FORMATION_NODE_FEAT_DIM
        self.observation_space = [Box(-inf, inf, (No,)) for _ in range(N)]          # environment.py:117-120, :781-813
        self.share_observation_space = [Box(-inf, inf, (No * N,)) for _ in range(N)]
        self.action_space = [Discrete(5) for _ in range(N)]
        self.node_observation_space = [Box(-inf, inf, (E, Nn)) for _ in range(N)]
        self.adj_observation_space = [Box(-inf, inf, (E, E)) for _ in range(N)]
        self.edge_observation_space = [Box(-inf, inf, (1,)) for _ in range(N)]
        self.agent_id_observation_space = [Box(-inf, inf, (1,)) for _ in range(N)]
        self.share_agent_id_observation_space = [Box(-inf, inf, (N,)) for _ in range(N)]
        self._out = self._outs[0]
        if episode_stats:
            _lib.check(self.lib.fm_formation_stats_enable(self._h, 1, self._stream()), "fm_formation_stats_enable")

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def _check_out(self, out: Dict[str, Any], with_step: bool) -> Dict[str, Any]:
        """Caller-owned output arrays: contiguous CUDA tensors of the API shapes on this env's device, ``adj`` one matrix
        per env ``[B,E,E]``.  Returns them under the keys of the result dicts, with the env's own info rows."""
        t, B, N, E = self.torch, self.num_envs, self.num_agents, self.num_entities
        want = {"obs": ((B, N, _lib.FORMATION_OBS_DIM), t.float32), "node_obs": ((B, N, E, _lib.FORMATION_NODE_FEAT_DIM), t.float32),
                "adj": ((B, E, E), t.float32)}
        if with_step:
            want.update(reward=((B, N), t.float32), done=((B, N), t.uint8))
        views = {}
        for name, (shape, dt) in want.items():
            x = out.get(name)
            if x is None or tuple(x.shape) != shape or x.dtype != dt or not x.is_contiguous() or x.device != self.device:
                raise ValueError(f"out[{name!r}] must be a contiguous {dt} tensor of shape {shape} on {self.device}")
            views["adj_env" if name == "adj" else name] = x
        if with_step:
            views["info"] = self._slots[0]["info"]
        return views

    @staticmethod
    def _outputs(views: Dict[str, Any]) -> _lib.FmOutputs:
        return _lib.FmOutputs(*[views[k].data_ptr() if k in views else None
                                for k in ("obs", "node_obs", "adj_env", "reward", "done", "info")])

    def reset_tensor(self, mask=None, out: Optional[Dict[str, Any]] = None) -> Dict[str, Any]:
        """Reset all envs (or those with ``mask`` != 0, [B]); returns ``obs``, ``node_obs``, ``adj_env``.  ``out``: write
        into the caller's ``obs [B,N,11]``, ``node_obs [B,N,E,13]``, ``adj [B,E,E]`` instead of the env's buffers."""
        t = self.torch
        views = self._check_out(out, with_step=False) if out is not None else None
        m = None
        if mask is not None:
            m = t.as_tensor(np.asarray(mask) if not t.is_tensor(mask) else mask).to(device=self.device, dtype=t.uint8).contiguous()
            if tuple(m.shape) != (self.num_envs,):
                raise ValueError(f"mask must have shape ({self.num_envs},)")
        o = self._outputs(views) if views is not None else self._out
        _lib.check(self.lib.fm_formation_reset(self._h, m.data_ptr() if m is not None else None, C.byref(o),
                                               self._stream()), "fm_formation_reset")
        if m is not None:
            t.cuda.current_stream(self.device).synchronize()          # keep `m` alive until consumed
        return dict(views) if views is not None else {k: self._buf[k] for k in ("obs", "node_obs", "adj_env")}

    def step_tensor(self, actions, out: Optional[Dict[str, Any]] = None) -> Dict[str, Any]:
        """One step; ``actions`` int32 CUDA ``[B,N]``.  ``out``: write into the caller's ``obs``, ``node_obs``,
        ``adj [B,E,E]``, ``reward [B,N]`` float32 and ``done [B,N]`` uint8 (the slabs ``DeviceRolloutBuffer.env_views``
        hands out) instead of the next slot of the ring, which then does not advance.  Same keys either way."""
        t = self.torch
        if not (t.is_tensor(actions) and actions.is_cuda and actions.dtype == t.int32 and actions.is_contiguous()
                and tuple(actions.shape) == (self.num_envs, self.num_agents)):
            raise ValueError(f"actions must be a contiguous int32 CUDA tensor [{self.num_envs},{self.num_agents}]")
        if out is not None:
            res = self._check_out(out, with_step=True)
            o = self._outputs(res)
        else:
            self._slot = (self._slot + 1) % len(self._slots)
            self._buf, self._out = self._slots[self._slot], self._outs[self._slot]
            res, o = dict(self._buf), self._out
        _lib.check(self.lib.fm_formation_step(self._h, actions.data_ptr(), C.byref(o), self._stream()),
                   "fm_formation_step")
        res["done"] = res["done"].view(t.bool)
        return res

    def read_stats(self, clear: bool = False, out=None):
        """Local episode-statistics vector (float64 CUDA tensor [15N+2], the layout of ``fm_stats_read``; see
        ``sharding.stats_layout`` / ``EpisodeStats``).  Needs ``episode_stats=True``.  ``out``: reuse a tensor."""
        t = self.torch
        if out is None:
            out = t.empty(self.lib.fm_stats_len(self.num_agents), dtype=t.float64, device=self.device)
        _lib.check(self.lib.fm_formation_stats_read(self._h, out.data_ptr(), int(clear), self._stream()), "fm_formation_stats_read")
        return out

    def rollout_tensor(self, actions):
        """T consecutive steps with pre-generated actions int32 CUDA ``[T, B, N]`` in ONE ``fm_formation_step_many`` call
        (``FM_FORM_LANES=2``: two env-range lanes on two streams).  Step t writes the output slot ``slots[t]`` of the ring (``num_slots`` sets,
        round robin: with T > num_slots the early steps are overwritten); returns ``slots``.  ``slot_outputs(k)`` are the
        tensors of slot k."""
        t = self.torch
        if not (t.is_tensor(actions) and actions.is_cuda and actions.dtype == t.int32 and actions.is_contiguous()
                and actions.dim() == 3 and tuple(actions.shape[1:]) == (self.num_envs, self.num_agents)):
            raise ValueError(f"actions must be a contiguous int32 CUDA tensor [T,{self.num_envs},{self.num_agents}]")
        T = int(actions.shape[0])
        slots = [(self._slot + 1 + k) % len(self._slots) for k in range(T)]
        outs = (_lib.FmOutputs * max(T, 1))(*[self._outs[k] for k in slots])
        _lib.check(self.lib.fm_formation_step_many(self._h, actions.data_ptr(), T, outs, self._stream()), "fm_formation_step_many")
        if T:
            self._slot = slots[-1]
            self._buf, self._out = self._slots[self._slot], self._outs[self._slot]
        return slots

    def slot_outputs(self, k: int) -> Dict[str, Any]:
        out = dict(self._slots[k])
        out["done"] = self._slots[k]["done"].view(self.torch.bool)
        return out

    # ------------------------------------------------------------------ ShareVecEnv interface (numpy)
    def reset(self):
        """``(obs, agent_id, node_obs, adj)`` (env_wrappers.py:997-1002)."""
        out = self.reset_tensor()
        return share_vec_env_tuple({k: v.cpu().numpy() for k, v in out.items()})

    def step(self, actions_env):
        """``(obs, agent_id, node_obs, adj, rewards [B,N], dones [B,N] bool, infos)`` (env_wrappers.py:983-996), auto-reset
        included when every agent of an env is done (:859-865)."""
        t = self.torch
        idx = decode_onehot_actions(actions_env, self.num_envs, self.num_agents)
        out = self.step_tensor(t.as_tensor(idx, dtype=t.int32).to(self.device))
        return share_vec_env_tuple({k: v.cpu().numpy() for k, v in out.items()}, self.cfg.max_speed is not None)

    def step_async(self, actions_env):
        self._pending = self.step(actions_env)

    def step_wait(self):
        r, self._pending = self._pending, None
        return r

    def render(self, mode: str = "human"):
        raise NotImplementedError("rendering is out of scope (SURVEY.md section 2, row 15)")

    # ------------------------------------------------------------------ state
    def _shapes(self):
        B, N, O, W = self.num_envs, self.num_agents, self.cfg.num_obstacles, self.cfg.num_walls
        per = {"pos": (B, N, 2), "vel": (B, N, 2), "landmark_pos": (B, N, 2), "obstacle_pos": (B, O, 2),
               "dist_traveled_mean": (B,), "dist_traveled_stddev": (B,), "step": (B,), "episode": (B,),
               "wall_axis": (B, W), "wall_orient": (B, W), "wall_len": (B,) if W else (0,)}
        return {name: per.get(name, (B, N)) for name in _lib.FORMATION_STATE_FIELDS}

    def _dtype(self, name):
        t = self.torch
        return t.int32 if name in _lib.FORMATION_STATE_INT_FIELDS else (t.uint8 if name == "status" else t.float32)

    def _struct(self, tensors) -> _lib.FmFormationState:
        st = _lib.FmFormationState()
        for name in _lib.FORMATION_STATE_FIELDS:
            v = tensors.get(name)
            setattr(st, name, v.data_ptr() if v is not None and v.numel() else None)
        return st

    def get_state(self) -> Dict[str, Any]:
        tensors = {n: self.torch.empty(sh, dtype=self._dtype(n), device=self.device) for n, sh in self._shapes().items()}
        st = self._struct(tensors)
        _lib.check(self.lib.fm_formation_get_state(self._h, C.byref(st), self._stream()), "fm_formation_get_state")
        return tensors

    def set_state(self, state: Dict[str, Any]) -> None:
        t, shapes, tensors = self.torch, self._shapes(), {}
        for name, v in state.items():
            if name not in shapes:
                raise KeyError(name)
            x = t.as_tensor(np.asarray(v) if not t.is_tensor(v) else v).to(device=self.device, dtype=self._dtype(name)).contiguous()
            if tuple(x.shape) != shapes[name]:
                raise ValueError(f"state[{name!r}] must have shape {shapes[name]}, got {tuple(x.shape)}")
            tensors[name] = x
        st = self._struct(tensors)
        _lib.check(self.lib.fm_formation_set_state(self._h, C.byref(st), self._stream()), "fm_formation_set_state")
        t.cuda.current_stream(self.device).synchronize()              # keep `tensors` alive until consumed

    def close(self) -> None:
        if self.closed:
            return
        self.torch.cuda.synchronize(self.device)
        self.lib.fm_formation_destroy(self._h)
        self._h, self.closed = None, True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
