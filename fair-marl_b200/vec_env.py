"""``B200GraphVecEnv``: device-resident, batched replacement of the reference's GraphMPE vector env.

Replaces, behind the same interface, the stack
``GraphSubprocVecEnv`` (onpolicy/envs/env_wrappers.py:951-1025) -> ``graphworker`` (:850-893) ->
``GraphMPEEnv`` (multiagent/MPE_env.py:55-77) -> ``MultiAgentGraphEnv`` (multiagent/environment.py:719-908)
-> ``World`` (multiagent/core.py:131-503) + ``navigation_graph.Scenario`` + ``marl_fair_assign``.

Two call styles:

* the reference API -- ``reset()`` / ``step(actions_env)`` with numpy in, numpy out (host buffers,
  one ``fm_step_host`` C-ABI call per step, which moves actions H2D and results D2H);
* the tensor fast path -- ``reset_tensor()`` / ``step_tensor(actions)`` with CUDA tensors in and
  out, no host synchronisation, outputs written into a ring of rollout slabs.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Any, Dict, List, Optional, Sequence

import numpy as np

from fair_marl_b200 import _lib
from fair_marl_b200.config import SimConfig
from fair_marl_b200.spaces import Box, Discrete


class _Nvtx:
    """NVTX ranges around the entry points (``FM_NVTX=1``): ``fm:reset``, ``fm:step``, ``fm:rollout``, ``fm:edge_list``,
    ``fm:step_host`` show up on the nsys / ncu timeline next to the kernels they launch (SURVEY.md section 5.1)."""
    enabled = __import__("os").environ.get("FM_NVTX", "0") not in ("", "0")

    def __init__(self, name: str):
        self.name = name

    def __enter__(self):
        if _Nvtx.enabled:
            import torch
            torch.cuda.nvtx.range_push(self.name)

    def __exit__(self, *exc):
        if _Nvtx.enabled:
            import torch
            torch.cuda.nvtx.range_pop()
        return False


class LazyInfos(Sequence):
    """``infos`` as the reference returns it -- a length-B sequence of length-N lists of dicts
    (env_wrappers.py:988-996) -- materialised from the device info rows only when indexed
    (the runner touches it at log time only, graph_mpe_runner.py:143-146)."""

    def __init__(self, env: "B200GraphVecEnv", version: int, fresh=None):
        # fresh: [B] bool, envs whose info rows were written by THIS step (the kernels write them on the step every agent
        # is done, or on every step with SimConfig.info_every_step); None = all of them
        self._env, self._version, self._rows, self._fresh = env, version, None, fresh

    def _fetch(self) -> np.ndarray:
        if self._rows is None:
            if self._env._step_version != self._version:
                raise RuntimeError("infos of an earlier step were not read before the next step()")
            self._rows = self._env._read_info_rows()
        return self._rows

    def __len__(self) -> int:
        return self._env.num_envs

    def __getitem__(self, b):
        if isinstance(b, slice):
            return [self[i] for i in range(*b.indices(len(self)))]
        if self._fresh is not None and not bool(self._fresh[b]):
            raise RuntimeError("info rows are written on terminal steps only; construct the env with "
                               "SimConfig(info_every_step=True) to read infos on every step (eval / render loops)")
        rows = self._fetch()[b]
        keys = _lib.INFO_KEYS if self._env.cfg.max_speed is not None else _lib.INFO_KEYS[:-1]
        return [{k: float(rows[i, j]) for j, k in enumerate(keys)} for i in range(rows.shape[0])]

    def as_array(self) -> np.ndarray:
        """[B, N, 14] float32, columns in ``INFO_KEYS`` order (rows of envs that were not terminal at this step hold the
        values of their last terminal step unless ``info_every_step`` is set)."""
        return self._fetch()


def make_spaces(num_agents: int, num_entities: int, node_feat_dim: int = _lib.NODE_FEAT_DIM, obs_dim: int = _lib.OBS_DIM) -> Dict[str, list]:
    """The per-agent space lists ``GMPERunner`` / ``GraphReplayBuffer`` read from the vec env (environment.py:117-190,
    :781-813; env_wrappers.py:951-980), as ``Box`` / ``Discrete`` stand-ins (``gym`` is not a dependency)."""
    N, E, inf = num_agents, num_entities, float("inf")
    return {
        "observation_space": [Box(-inf, inf, (obs_dim,)) for _ in range(N)],
        "share_observation_space": [Box(-inf, inf, (obs_dim * N,)) for _ in range(N)],
        "action_space": [Discrete(5) for _ in range(N)],
        "node_observation_space": [Box(-inf, inf, (E, node_feat_dim)) for _ in range(N)],
        "adj_observation_space": [Box(-inf, inf, (E, E)) for _ in range(N)],
        "edge_observation_space": [Box(-inf, inf, (1,)) for _ in range(N)],
        "agent_id_observation_space": [Box(-inf, inf, (1,)) for _ in range(N)],
        "share_agent_id_observation_space": [Box(-inf, inf, (N,)) for _ in range(N)],
    }


class B200GraphVecEnv:
    """ShareVecEnv-compatible batched ``navigation_graph`` simulator on one B200.

    Parameters
    ----------
    args : the reference's ``all_args`` Namespace (fields listed in ``SimConfig``) or a ``SimConfig``.
    num_envs : envs on THIS device (default ``args.n_rollout_threads``).
    device : CUDA device index.
    seed : base seed (default ``args.seed``); reset streams are keyed by (seed, global env index).
    env_offset : global index of local env 0 when the batch is sharded over ranks.
    num_slots : rollout slabs for the tensor path (``step_tensor`` writes slot (t+1) % num_slots).
    dummy_vec_env : mirror ``GraphDummyVecEnv`` (env_wrappers.py:895-950) instead of ``GraphSubprocVecEnv``:
        ``step()`` returns the 8-tuple ``(..., infos, reset_count)`` with ``reset_count = 1`` when an env finished
        its episode in this step (the eval / render loops read it, graph_mpe_runner.py:684-685).
    """

    closed = False

    def __init__(self, args: Any = None, num_envs: Optional[int] = None, device: int = 0,
                 seed: Optional[int] = None, env_offset: int = 0, num_slots: int = 2, dummy_vec_env: bool = False,
                 **overrides):
        torch = _lib.require_cuda()
        self.torch = torch
        self.lib = _lib.load()
        self.cfg = args if isinstance(args, SimConfig) else SimConfig.from_args(args if args is not None else object(), **overrides)
        if num_envs is None:
            num_envs = getattr(args, "n_rollout_threads", None)
        if not num_envs or num_envs <= 0:
            raise ValueError("num_envs must be given (or args.n_rollout_threads)")
        if seed is None:
            seed = getattr(args, "seed", 1)
        self.num_envs = int(num_envs)
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        self.seed = int(seed)
        self.env_offset = int(env_offset)
        cfg = self.cfg
        N, E = cfg.num_agents, cfg.num_entities
        self.num_agents, self.num_entities = N, E
        self.node_feat_dim = cfg.node_feat_dim

        c = _lib.FmConfig(
            num_envs=self.num_envs, num_agents=N, num_obstacles=cfg.num_obstacles,
            episode_length=cfg.episode_length, env_offset=self.env_offset, seed=self.seed & (2 ** 64 - 1),
            world_size=cfg.world_size, max_speed=(cfg.max_speed if cfg.max_speed is not None else 0.0),
            collision_rew=cfg.collision_rew, goal_rew=cfg.goal_rew, min_dist_thresh=cfg.min_dist_thresh,
            fair_rew=cfg.fair_rew, zeroshift=cfg.zeroshift, max_edge_dist=cfg.max_edge_dist,
            fairness_reward=int(cfg.fairness_reward), collaborative=int(cfg.collaborative),
            auto_reset=int(cfg.auto_reset), info_every_step=int(cfg.info_every_step),
            mapping={"auto": 0, "group": 1, "aw": 2}[cfg.mapping],
            graph_feat_global=int(cfg.graph_feat_type == "global"), num_walls=int(cfg.num_walls))
        self._h = C.c_void_p()
        _lib.check(self.lib.fm_create(C.byref(c), self.device_index, C.byref(self._h)), "fm_create")

        # spaces (environment.py:117-190, :781-813)
        for name, spaces in make_spaces(N, E, self.node_feat_dim).items():
            setattr(self, name, spaces)

        # get_id (navigation_graph.py:875-876): global_id == agent index
        self._agent_id_host = np.tile(np.arange(N, dtype=np.int64)[None, :, None], (self.num_envs, 1, 1))
        self._agent_id_dev = None
        self._host = None               # pinned host buffers for the numpy API
        self._slabs = None              # device rollout slabs for the tensor API
        self.num_slots = int(num_slots)
        self._slot = 0
        self._step_version = 0
        self._pending_actions = None
        self._last_step_api = None
        self._plans = {}
        self.dummy_vec_env = bool(dummy_vec_env)

    # ------------------------------------------------------------------ helpers
    def _stream(self) -> int:
        return self.torch.cuda.current_stream(self.device).cuda_stream

    def _ensure_host(self):
        if self._host is None:
            t, B, N, E = self.torch, self.num_envs, self.num_agents, self.num_entities
            pin = dict(pin_memory=True)
            self._host = {
                "onehot": t.empty((B, N, 5), dtype=t.float32, **pin),
                "obs": [t.empty((B, N, _lib.OBS_DIM), dtype=t.float32, **pin) for _ in range(2)],
                "node_obs": [t.empty((B, N, E, self.node_feat_dim), dtype=t.float32, **pin) for _ in range(2)],
                "adj": [t.empty((B, E, E), dtype=t.float32, **pin) for _ in range(2)],
                "reward": [t.empty((B, N), dtype=t.float32, **pin) for _ in range(2)],
                "done": [t.empty((B, N), dtype=t.uint8, **pin) for _ in range(2)],
                "info": t.empty((B, N, _lib.INFO_DIM), dtype=t.float32, **pin),
                "flip": 0,
            }
            # env-range lanes of the host step (FM_HOST_LANES overrides; the persistent kernel has no ranged launch)
            lanes = int(os.environ.get("FM_HOST_LANES", "4" if B >= 16384 else "1"))
            lanes = 1 if os.environ.get("FM_ROLL", "0") not in ("", "0") else max(1, min(8, lanes))
            self._host_lanes, self._host_lane_bounds = lanes, []
            for k in range(lanes):
                b0, b1 = C.c_int32(), C.c_int32()
                _lib.check(self.lib.fm_host_lane_range(self._h, k, lanes, C.byref(b0), C.byref(b1)), "fm_host_lane_range")
                self._host_lane_bounds.append((b0.value, b1.value))
        return self._host

    def _ensure_slabs(self):
        if self._slabs is None:
            t, B, N, E, S = self.torch, self.num_envs, self.num_agents, self.num_entities, self.num_slots
            kw = dict(device=self.device)
            self._slabs = {
                "obs": t.empty((S, B, N, _lib.OBS_DIM), dtype=t.float32, **kw),
                "node_obs": t.empty((S, B, N, E, self.node_feat_dim), dtype=t.float32, **kw),
                "adj": t.empty((S, B, E, E), dtype=t.float32, **kw),
                "reward": t.empty((S, B, N), dtype=t.float32, **kw),
                "done": t.empty((S, B, N), dtype=t.uint8, **kw),
                "info": t.zeros((B, N, _lib.INFO_DIM), dtype=t.float32, **kw),
            }
            self._agent_id_dev = t.arange(N, dtype=t.int32, device=self.device)[None, :, None].expand(B, N, 1)
        return self._slabs

    def _outputs_struct(self, tensors: Dict[str, Any], with_step: bool) -> _lib.FmOutputs:
        o = _lib.FmOutputs()
        o.obs = tensors["obs"].data_ptr()
        o.node_obs = tensors["node_obs"].data_ptr()
        o.adj = tensors["adj"].data_ptr()
        if with_step:
            o.reward = tensors["reward"].data_ptr()
            o.done = tensors["done"].data_ptr()
            if tensors.get("info") is not None:
                o.info = tensors["info"].data_ptr()
        return o

    def _package(self, slot: int, with_step: bool) -> Dict[str, Any]:
        s, B, N, E = self._slabs, self.num_envs, self.num_agents, self.num_entities
        out = {"obs": s["obs"][slot], "node_obs": s["node_obs"][slot],
               "adj": s["adj"][slot][:, None].expand(B, N, E, E),      # written once per env
               "adj_env": s["adj"][slot], "agent_id": self._agent_id_dev, "slot": slot}
        if with_step:
            out.update(reward=s["reward"][slot], done=s["done"][slot].view(self.torch.bool), info=s["info"])   # zero-copy
        return out

    # ------------------------------------------------------------------ tensor fast path
    def _check_out(self, out: Dict[str, Any], with_step: bool) -> Dict[str, Any]:
        """Validate caller-owned output arrays (e.g. slabs of a ``DeviceRolloutBuffer``): contiguous CUDA tensors of the
        API shapes; ``adj`` is ``[B, E, E]`` (one matrix per env)."""
        t, B, N, E = self.torch, self.num_envs, self.num_agents, self.num_entities
        want = {"obs": ((B, N, _lib.OBS_DIM), t.float32), "node_obs": ((B, N, E, self.node_feat_dim), t.float32),
                "adj": ((B, E, E), t.float32)}
        if with_step:
            want.update(reward=((B, N), t.float32), done=((B, N), t.uint8))
        views = {}
        for name, (shape, dt) in want.items():
            x = out.get(name)
            if x is None or tuple(x.shape) != shape or x.dtype != dt or not x.is_contiguous() or x.device != self.device:
                raise ValueError(f"out[{name!r}] must be a contiguous {dt} tensor of shape {shape} on {self.device}")
            views[name] = x
        return views

    def _package_out(self, views: Dict[str, Any], with_step: bool) -> Dict[str, Any]:
        B, N, E = self.num_envs, self.num_agents, self.num_entities
        self._ensure_slabs()
        res = {"obs": views["obs"], "node_obs": views["node_obs"], "adj": views["adj"][:, None].expand(B, N, E, E),
               "adj_env": views["adj"], "agent_id": self._agent_id_dev, "slot": None}
        if with_step:
            res.update(reward=views["reward"], done=views["done"].view(self.torch.bool), info=self._slabs["info"])
        return res

    def reset_tensor(self, mask=None, out: Optional[Dict[str, Any]] = None) -> Dict[str, Any]:
        """Reset envs (all, or those with ``mask`` != 0: uint8 CUDA tensor [B]); returns device tensors
        ``obs [B,N,7]``, ``node_obs [B,N,E,11]``, ``adj [B,N,E,E]`` (stride-0 view), ``agent_id``.
        ``out``: caller-owned arrays to write into instead of the env's slab ring (see ``_check_out``)."""
        s = self._ensure_slabs()
        slot = self._slot
        views = self._check_out(out, with_step=False) if out is not None else {k: s[k][slot] for k in ("obs", "node_obs", "adj")}
        o = self._outputs_struct(views, with_step=False)
        mptr = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=self.torch.uint8).contiguous()
            mptr = mask.data_ptr()
        with _Nvtx("fm:reset"):
            _lib.check(self.lib.fm_reset(self._h, mptr, C.byref(o), self._stream()), "fm_reset")
        return self._package_out(views, with_step=False) if out is not None else self._package(slot, with_step=False)

    def observe_tensor(self, out: Optional[Dict[str, Any]] = None) -> Dict[str, Any]:
        """Observation of the current state without stepping or resetting (``fm_observe``)."""
        s = self._ensure_slabs()
        slot = self._slot
        views = self._check_out(out, with_step=False) if out is not None else {k: s[k][slot] for k in ("obs", "node_obs", "adj")}
        o = self._outputs_struct(views, with_step=False)
        _lib.check(self.lib.fm_observe(self._h, C.byref(o), self._stream()), "fm_observe")
        return self._package_out(views, with_step=False) if out is not None else self._package(slot, with_step=False)

    def observe_soa_tensor(self) -> Dict[str, Any]:
        """The observation of the current state in the SoA layout (``fm_observe_soa``): one plane per value, envs fastest --
        ``obs [N, 7, B]``, ``node_obs [N, E, F, B]``, ``adj [E, E, B]`` (views of buffers whose env stride is
        ``fm_soa_stride``; bit-identical to ``observe_tensor`` transposed).  For device-side consumers with lane = env."""
        t = self.torch
        N, E, B = self.num_agents, self.num_entities, self.num_envs
        F = _lib.NODE_FEAT_DIM_GLOBAL if self.cfg.graph_feat_type == "global" else _lib.NODE_FEAT_DIM
        S = int(self.lib.fm_soa_stride(self._h))
        if getattr(self, "_soa", None) is None:
            f32 = dict(dtype=t.float32, device=self.device)
            self._soa = {"obs": t.empty((N, _lib.OBS_DIM, S), **f32), "node_obs": t.empty((N, E, F, S), **f32), "adj": t.empty((E, E, S), **f32)}
        o = _lib.FmSoaOutputs(self._soa["obs"].data_ptr(), self._soa["node_obs"].data_ptr(), self._soa["adj"].data_ptr())
        _lib.check(self.lib.fm_observe_soa(self._h, C.byref(o), self._stream()), "fm_observe_soa")
        return {k: v[..., :B] for k, v in self._soa.items()}

    def check_finite(self):
        """``(flags [B] int32, count [1] int32)`` device tensors: envs whose dynamic state holds a NaN / Inf (``fm_check_finite``)."""
        t = self.torch
        flags = t.empty((self.num_envs,), dtype=t.int32, device=self.device)
        count = t.empty((1,), dtype=t.int32, device=self.device)
        _lib.check(self.lib.fm_check_finite(self._h, flags.data_ptr(), count.data_ptr(), self._stream()), "fm_check_finite")
        return flags, count

    def step_tensor(self, actions, out: Optional[Dict[str, Any]] = None) -> Dict[str, Any]:
        """One env step.  ``actions``: int32 CUDA tensor [B, N] in {0..4}, or float32 [B, N, 5] one-hot.
        Asynchronous on the current stream; the returned tensors are views of slab ``slot``, or of ``out`` when the
        caller passes its own arrays (``obs``, ``node_obs``, ``adj [B,E,E]``, ``reward``, ``done``: e.g. slab t + 1 of a
        ``DeviceRolloutBuffer``, so that the step kernel writes the rollout buffer directly)."""
        t = self.torch
        s = self._ensure_slabs()
        if out is not None:
            views = self._check_out(out, with_step=True)
            views["info"] = s["info"]
            o = self._outputs_struct(views, with_step=True)
            result = None
        else:
            self._slot = slot = (self._slot + 1) % self.num_slots
            cached = self._plans.get(("slot", slot))
            if cached is None:                      # FmOutputs struct and result views of a ring slot are built once
                views = {k: s[k][slot] for k in ("obs", "node_obs", "adj", "reward", "done")}
                views["info"] = s["info"]
                cached = self._plans[("slot", slot)] = (self._outputs_struct(views, with_step=True), self._package(slot, with_step=True))
            o, result = cached
        B, N = self.num_envs, self.num_agents
        with _Nvtx("fm:step"):
            if actions.dim() == 2:
                if actions.dtype != t.int32 or not actions.is_contiguous() or actions.shape != (B, N):
                    actions = actions.to(t.int32).contiguous().view(B, N)
                rc = self.lib.fm_step(self._h, actions.data_ptr(), C.byref(o), self._stream())
            else:
                if actions.dtype != t.float32 or not actions.is_contiguous() or actions.shape != (B, N, 5):
                    actions = actions.to(t.float32).contiguous().view(B, N, 5)
                rc = self.lib.fm_step_onehot(self._h, actions.data_ptr(), C.byref(o), self._stream())
        _lib.check(rc, "fm_step")
        self._step_version += 1
        self._last_step_api = "tensor"
        return self._package_out(views, with_step=True) if result is None else dict(result)

    def edge_list_tensor(self, adj_env, repeat: int = 1, inclusive: bool = False) -> Dict[str, Any]:
        """Policy-side edge list of ``adj_env [B,E,E]`` (``process_adj``, gnn_new.py:381-413) WITHOUT a host sync:
        buffers of worst-case capacity are allocated once and reused; ``nnz`` stays on the device.  Returns
        ``edge_index [2, capacity]`` (int64, the first ``nnz`` columns are valid, (b, i, j) order, node ids offset by
        ``b*E``), ``edge_attr [capacity]``, ``offsets [B*repeat + 1]`` and ``nnz [1]``.  ``repeat=N`` emits every
        env's graph once per agent, i.e. the batch the policy sees.  ``fair_marl_b200.process_adj`` is the
        synchronising variant that trims to ``nnz``."""
        t, B, E = self.torch, self.num_envs, self.num_entities
        if tuple(adj_env.shape) != (B, E, E) or adj_env.dtype != t.float32 or not adj_env.is_contiguous():
            raise ValueError(f"adj_env must be a contiguous float32 tensor of shape {(B, E, E)}")
        key = ("edges", repeat)
        buf = self._plans.get(key)
        if buf is None:
            cap = B * repeat * E * (E - 1)          # adj_env is a distance matrix: zero diagonal
            buf = self._plans[key] = {
                "capacity": cap,
                "offsets": t.empty(B * repeat + 1, dtype=t.int64, device=self.device),
                "edge_index": t.empty((2, max(cap, 1)), dtype=t.int64, device=self.device),
                "edge_attr": t.empty(max(cap, 1), dtype=t.float32, device=self.device),
                "nnz": t.zeros(1, dtype=t.int64, device=self.device)}
        _lib.check(self.lib.fm_edge_list(self.device_index, adj_env.data_ptr(), B, E, float(self.cfg.max_edge_dist),
                                         int(inclusive), int(repeat), buf["capacity"], buf["offsets"].data_ptr(),
                                         buf["edge_index"].data_ptr(), buf["edge_attr"].data_ptr(), buf["nnz"].data_ptr(),
                                         self._stream()), "fm_edge_list")
        return buf

    def rollout_tensor(self, actions) -> List[int]:
        """``T`` consecutive steps from one host call (``fm_step_many``): ``actions`` int32 CUDA tensor
        [T, B, N].  Step t writes slab slot (slot + 1 + t) % num_slots; returns the slot of every step.
        Asynchronous; no per-step Python or ctypes overhead."""
        t = self.torch
        s = self._ensure_slabs()
        B, N = self.num_envs, self.num_agents
        if actions.dtype != t.int32 or not actions.is_contiguous() or actions.dim() != 3 or actions.shape[1:] != (B, N):
            raise ValueError("actions must be a contiguous int32 CUDA tensor [T, B, N]")
        T = int(actions.shape[0])
        if T == 0:
            return []
        S = self.num_slots
        start = (self._slot + 1) % S
        # One FmOutputs table for the slab ring, repeated often enough that any (start slot, T) is a contiguous run of
        # it: a rollout call does no per-step Python work (no tensor slicing, no data_ptr(), no struct filling).
        reps = (S - 1 + T + S - 1) // S
        ring = self._plans.get("ring")
        if ring is None or ring[1] < reps:
            arr = (_lib.FmOutputs * (S * reps))()
            for k in range(S):
                views = {name: s[name][k] for name in ("obs", "node_obs", "adj", "reward", "done")}
                views["info"] = s["info"]
                o = self._outputs_struct(views, with_step=True)
                for r in range(reps):
                    arr[r * S + k] = o
            ring = self._plans["ring"] = (arr, reps)
        arr = ring[0]
        first = C.cast(C.addressof(arr) + start * C.sizeof(_lib.FmOutputs), C.POINTER(_lib.FmOutputs))
        slots = [(start + k) % S for k in range(T)]
        with _Nvtx("fm:rollout"):
            _lib.check(self.lib.fm_step_many(self._h, actions.data_ptr(), T, first, self._stream()), "fm_step_many")
        self._slot = slots[-1] if slots else self._slot
        self._step_version += T
        self._last_step_api = "tensor"
        return slots

    def slot_outputs(self, slot: int) -> Dict[str, Any]:
        """Views of rollout slab ``slot`` (as returned by ``step_tensor``)."""
        self._ensure_slabs()
        return self._package(slot, with_step=True)

    # ------------------------------------------------------------------ reference (numpy) API
    def _host_outputs(self, with_step: bool):
        h = self._ensure_host()
        h["flip"] ^= 1
        f = h["flip"]
        cur = {k: h[k][f] for k in ("obs", "node_obs", "adj", "reward", "done")}
        o = _lib.FmOutputs()
        o.obs, o.node_obs, o.adj = cur["obs"].data_ptr(), cur["node_obs"].data_ptr(), cur["adj"].data_ptr()
        if with_step:
            o.reward, o.done = cur["reward"].data_ptr(), cur["done"].data_ptr()
        return cur, o

    def _numpy_obs(self, cur, copy: bool):
        B, N, E = self.num_envs, self.num_agents, self.num_entities
        obs, node, adj = cur["obs"].numpy(), cur["node_obs"].numpy(), cur["adj"].numpy()
        if copy:
            obs, node, adj = obs.copy(), node.copy(), adj.copy()
        adj_n = np.broadcast_to(adj[:, None], (B, N, E, E))     # same matrix for the N agents of an env
        return obs, self._agent_id_host, node, adj_n

    def reset(self, copy: bool = False):
        """``(obs [B,N,7], agent_id [B,N,1], node_obs [B,N,E,11], adj [B,N,E,E])`` as numpy
        (env_wrappers.py:997-1002).  Arrays are views of pinned double buffers (valid until the call
        after next) unless ``copy=True``."""
        cur, o = self._host_outputs(with_step=False)
        _lib.check(self.lib.fm_reset_host(self._h, None, C.byref(o), self._stream()), "fm_reset_host")
        return self._numpy_obs(cur, copy)

    def step_async(self, actions) -> None:
        self._pending_actions = actions

    def step_wait(self, copy: bool = False):
        actions = self._pending_actions
        self._pending_actions = None
        if actions is None:
            raise RuntimeError("step_wait() without step_async()")
        h = self._ensure_host()
        B, N = self.num_envs, self.num_agents
        a = np.asarray(actions)
        if a.shape == (B, N, 5):
            onehot = True
        elif a.shape in ((B, N), (B, N, 1)):                          # convenience: action indices
            onehot, a = False, a.reshape(B, N, 1).astype(np.int64)
        else:
            raise ValueError(f"actions must be [B,N,5] one-hot (or [B,N] indices), got {a.shape}")
        cur, o = self._host_outputs(with_step=True)
        oh = h["onehot"].numpy()
        # Large batches go as env-range lanes: the rows of lane k + 1 are converted into the pinned float32 buffer (the runner
        # hands float64 one-hot, graph_mpe_runner.py:429-431) while lane k's results cross the bus (fm_step_host_lane).
        lanes = self._host_lanes
        with _Nvtx("fm:step_host"):
            for k in range(lanes):
                b0, b1 = self._host_lane_bounds[k]
                if onehot:
                    oh[b0:b1] = a[b0:b1]                              # cast to float32 into pinned memory
                else:
                    oh[b0:b1] = 0.0
                    np.put_along_axis(oh[b0:b1], a[b0:b1], 1.0, axis=2)
                if lanes == 1:
                    _lib.check(self.lib.fm_step_host(self._h, h["onehot"].data_ptr(), C.byref(o), self._stream()), "fm_step_host")
                else:
                    _lib.check(self.lib.fm_step_host_lane(self._h, h["onehot"].data_ptr(), C.byref(o), k, lanes, self._stream()), "fm_step_host_lane")
        self._step_version += 1
        self._last_step_api = "host"
        obs, ag_id, node, adj_n = self._numpy_obs(cur, copy)
        rew = cur["reward"].numpy()
        done = cur["done"].numpy().astype(bool)
        if copy:
            rew = rew.copy()
        fresh = None if self.cfg.info_every_step else done.all(axis=1)
        if self.dummy_vec_env:                                        # env_wrappers.py:917-928
            reset_count = 1 if bool(done.all(axis=1).any()) else 0
            return obs, ag_id, node, adj_n, rew, done, LazyInfos(self, self._step_version, fresh), reset_count
        return obs, ag_id, node, adj_n, rew, done, LazyInfos(self, self._step_version, fresh)

    def step(self, actions, copy: bool = False):
        """``(obs, agent_id, node_obs, adj, rewards [B,N], dones [B,N] bool, infos)`` -- the 7-tuple of
        GraphSubprocVecEnv.step_wait (env_wrappers.py:988-996), auto-reset included (:859-865)."""
        self.step_async(actions)
        return self.step_wait(copy=copy)

    def _read_info_rows(self) -> np.ndarray:
        if self._last_step_api == "host":
            h = self._host
            _lib.check(self.lib.fm_read_info_host(self._h, h["info"].data_ptr(), self._stream()), "fm_read_info_host")
            return h["info"].numpy().copy()
        return self._slabs["info"].cpu().numpy()

    # ------------------------------------------------------------------ state, stats, misc
    def _state_struct(self, tensors: Dict[str, Any]) -> _lib.FmState:
        st = _lib.FmState()
        for name in _lib.STATE_FIELDS:
            v = tensors.get(name)
            setattr(st, name, v.data_ptr() if v is not None else None)
        return st

    def _state_shapes(self):
        B, N, O, W = self.num_envs, self.num_agents, self.cfg.num_obstacles, self.cfg.num_walls
        walls = {"wall_axis": (B, W), "wall_orient": (B, W), "wall_len": (B,)} if W else {}
        return {**walls, "pos": (B, N, 2), "vel": (B, N, 2), "p_dist": (B, N), "landmark_pos": (B, N, 2),
                "obstacle_pos": (B, O, 2), "goal_match": (B, N), "dists_to_goal": (B, N),
                "times_required": (B, N), "dist_left_to_goal": (B, N), "num_agent_collisions": (B, N),
                "num_obstacle_collisions": (B, N), "dist_traveled_mean": (B,), "dist_traveled_stddev": (B,),
                "step": (B,), "min_time": (B, N), "episode": (B,)}

    def get_state(self) -> Dict[str, Any]:
        """Full simulator state as CUDA tensors in API layout (float32 / int32)."""
        t = self.torch
        tensors = {}
        for name, shape in self._state_shapes().items():
            dt = t.int32 if name in _lib.STATE_INT_FIELDS else t.float32
            tensors[name] = t.empty(shape, dtype=dt, device=self.device)
        st = self._state_struct(tensors)
        _lib.check(self.lib.fm_get_state(self._h, C.byref(st), self._stream()), "fm_get_state")
        return tensors

    def set_state(self, state: Dict[str, Any]) -> None:
        """Inject (a subset of) the state; values may be numpy or tensors, cast to float32 / int32."""
        t = self.torch
        shapes = self._state_shapes()
        tensors = {}
        for name, v in state.items():
            if name not in shapes:
                raise KeyError(name)
            dt = t.int32 if name in _lib.STATE_INT_FIELDS else t.float32
            x = t.as_tensor(np.asarray(v) if not t.is_tensor(v) else v).to(device=self.device, dtype=dt).contiguous()
            if tuple(x.shape) != shapes[name]:
                raise ValueError(f"state[{name!r}] must have shape {shapes[name]}, got {tuple(x.shape)}")
            tensors[name] = x
        st = self._state_struct(tensors)
        _lib.check(self.lib.fm_set_state(self._h, C.byref(st), self._stream()), "fm_set_state")
        self.torch.cuda.current_stream(self.device).synchronize()      # keep `tensors` alive until consumed

    def read_stats(self, clear: bool = False, out=None):
        """Local episode-statistics vector (float64 CUDA tensor [15N+2]); see fm_stats_read.  ``out``: reuse a tensor."""
        t = self.torch
        if out is None:
            out = t.empty(self.lib.fm_stats_len(self.num_agents), dtype=t.float64, device=self.device)
        _lib.check(self.lib.fm_stats_read(self._h, out.data_ptr(), int(clear), self._stream()), "fm_stats_read")
        return out

    @property
    def mapping(self) -> str:
        """Kernel mapping in use: 'group' (group-per-env) or 'aw' (agent-warp)."""
        return {1: "group", 2: "aw"}[int(self.lib.fm_mapping(self._h))]

    @property
    def kernel_launches(self) -> int:
        n = C.c_int64()
        _lib.check(self.lib.fm_kernel_launches(self._h, C.byref(n)))
        return int(n.value)

    @property
    def algorithmic_bytes_per_step(self) -> int:
        return int(self.lib.fm_algorithmic_bytes_per_step(self._h))

    def render(self, mode: str = "human"):
        raise NotImplementedError("rendering is out of scope (SURVEY.md section 2, row 15)")

    def close(self) -> None:
        if self.closed:
            return
        self.torch.cuda.synchronize(self.device)
        self.lib.fm_destroy(self._h)
        self._h = None
        self.closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def make_train_env(all_args, device: int = 0, rank: int = 0, world_size: int = 1):
    """Drop-in for ``make_train_env`` in onpolicy/scripts/train_mpe.py:21-43 when
    ``env_name == 'GraphMPE'``: ``n_rollout_threads`` envs, sharded over ranks if world_size > 1.  The four formation
    scenarios (``formation.SCENARIO_MODES``) give a ``B200FormationVecEnv`` with its episode statistics on."""
    from fair_marl_b200.formation import SCENARIO_MODES, B200FormationVecEnv, FormationSimConfig
    from fair_marl_b200.sharding import shard_range
    if getattr(all_args, "env_name", "GraphMPE") != "GraphMPE":
        raise NotImplementedError(f"Can not support the {all_args.env_name} environment")
    off, cnt = shard_range(all_args.n_rollout_threads, world_size, rank)
    if getattr(all_args, "scenario_name", None) in SCENARIO_MODES:
        return B200FormationVecEnv(FormationSimConfig.from_args(all_args), num_envs=cnt, device=device, seed=all_args.seed,
                                   env_offset=off, episode_stats=True)
    return B200GraphVecEnv(all_args, num_envs=cnt, device=device, seed=all_args.seed, env_offset=off)
