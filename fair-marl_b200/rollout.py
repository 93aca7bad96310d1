"""Device-resident rollout buffer and collection loop (SURVEY.md N1; BASELINE config 5).

Replaces, for the data path of one rollout, the host-side

* ``GraphReplayBuffer`` storage / ``insert`` / ``after_update`` / ``compute_returns``
  (onpolicy/utils/graph_buffer.py:15-251, :253-268, :270-341), and
* ``GMPERunner.collect`` / ``insert`` and the step loop of ``GMPERunner.run``
  (onpolicy/runner/shared/graph_mpe_runner.py:60-80, :396-436, :438-488).

In the reference every step concatenates ``[B, N, ...]`` numpy arrays, copies them to the policy's device, and
copies the env outputs into the buffer (``.copy()`` per field).  Here the buffer slabs ARE the simulator's output
arrays: ``step_tensor(actions, out=buffer.env_views(t + 1))`` makes the fused step kernel write ``obs``,
``node_obs``, ``adj``, ``reward`` and ``done`` of step t straight into slab t + 1 (TMA bulk stores into the rollout
buffer, no intermediate copy); ``adj`` is kept once per env and exposed per agent as a stride-0 view, ``share_obs``
and ``share_agent_id`` are views too.  The policy forward reads the slabs in place; nothing touches the host.
"""
from __future__ import annotations

from typing import Any, Dict, Optional, Tuple

import torch


class DeviceRolloutBuffer:
    """``GraphReplayBuffer`` with torch tensors on one device.  Field names and shapes follow the reference
    (graph_buffer.py:70-165) except that ``adj`` is stored once per env (``adj_env [T+1, B, E, E]``; the reference
    stores the same matrix N times, navigation_graph.py:1033) and ``share_obs`` / ``share_agent_id`` are views."""

    def __init__(self, episode_length: int, num_envs: int, num_agents: int, num_entities: int, obs_dim: int = 7,
                 node_feat_dim: int = 11, hidden_size: int = 64, recurrent_N: int = 1, action_dim: int = 5,
                 gamma: float = 0.99, gae_lambda: float = 0.95, use_gae: bool = True, device: Any = "cuda",
                 use_proper_time_limits: bool = False):
        T, B, N, E = int(episode_length), int(num_envs), int(num_agents), int(num_entities)
        self.episode_length, self.n_rollout_threads, self.num_agents, self.num_entities = T, B, N, E
        self.gamma, self.gae_lambda, self._use_gae = gamma, gae_lambda, use_gae
        self._use_proper_time_limits = use_proper_time_limits
        self.device = torch.device(device)
        f32 = dict(dtype=torch.float32, device=self.device)
        self.obs = torch.zeros((T + 1, B, N, obs_dim), **f32)
        self.node_obs = torch.zeros((T + 1, B, N, E, node_feat_dim), **f32)
        self.adj_env = torch.zeros((T + 1, B, E, E), **f32)
        self.agent_id = torch.arange(N, dtype=torch.int32, device=self.device).view(1, 1, N, 1).expand(T + 1, B, N, 1)
        self.rnn_states = torch.zeros((T + 1, B, N, recurrent_N, hidden_size), **f32)
        self.rnn_states_critic = torch.zeros_like(self.rnn_states)
        self.value_preds = torch.zeros((T + 1, B, N, 1), **f32)
        self.returns = torch.zeros_like(self.value_preds)
        self.available_actions = torch.ones((1, 1, 1, action_dim), **f32).expand(T + 1, B, N, action_dim)
        self.actions = torch.zeros((T, B, N, 1), **f32)              # float32 like the reference (:139-143)
        self.actions_env = torch.zeros((T, B, N), dtype=torch.int32, device=self.device)   # what the simulator consumed
        self.action_log_probs = torch.zeros((T, B, N, 1), **f32)
        self.rewards = torch.zeros((T, B, N, 1), **f32)
        self.dones = torch.zeros((T, B, N), dtype=torch.uint8, device=self.device)
        self.masks = torch.ones((T + 1, B, N, 1), **f32)
        self.bad_masks = torch.ones_like(self.masks)
        self.active_masks = torch.ones_like(self.masks)
        self.step = 0
        self.advantage_stats: Optional[torch.Tensor] = None   # [2] (mean, std) of the last advantages() call

    # ---- views the reference materialises ------------------------------------------------------------------
    @property
    def adj(self) -> torch.Tensor:
        """[T+1, B, N, E, E], the env's matrix for each of its agents (stride 0 over N)."""
        T1, B, E, _ = self.adj_env.shape
        return self.adj_env.unsqueeze(2).expand(T1, B, self.num_agents, E, E)

    @property
    def share_obs(self) -> torch.Tensor:
        """[T+1, B, N, N*obs_dim]: all agents' observations, repeated per agent (graph_mpe_runner.py:470-473)."""
        T1, B, N, D = self.obs.shape
        return self.obs.reshape(T1, B, 1, N * D).expand(T1, B, N, N * D)

    @property
    def share_agent_id(self) -> torch.Tensor:
        T1, B, N, _ = self.agent_id.shape
        return self.agent_id.reshape(T1, B, 1, N).expand(T1, B, N, N)

    def env_views(self, t: int, with_step: bool = True) -> Dict[str, torch.Tensor]:
        """The arrays of slab ``t`` the simulator writes (``B200GraphVecEnv.step_tensor(out=...)``): the observation
        of time t, and -- for a step -- the reward / done of the transition t-1 -> t."""
        v = {"obs": self.obs[t], "node_obs": self.node_obs[t], "adj": self.adj_env[t]}
        if with_step:
            v["reward"] = self.rewards[t - 1].view(self.n_rollout_threads, self.num_agents)
            v["done"] = self.dones[t - 1]
        return v

    # ---- GraphReplayBuffer.insert (graph_buffer.py:168-251) + GMPERunner.insert (:438-488) -----------------
    def insert_policy(self, rnn_states: torch.Tensor, rnn_states_critic: torch.Tensor, actions: torch.Tensor,
                      action_log_probs: torch.Tensor, value_preds: torch.Tensor) -> None:
        """Policy-side fields of step ``self.step``; the env-side fields (obs, node_obs, adj, rewards, dones of the
        same step) have been written in place by the step kernel.  Masks and the RNN-state reset follow
        GMPERunner.insert: ``masks = 1 - done``; ``rnn_states[done] = 0``; ``active_masks`` is 1 where the agent is
        alive or the whole env is done."""
        t, B, N = self.step, self.n_rollout_threads, self.num_agents
        done = self.dones[t].bool()
        keep = (~done).to(torch.float32).view(B, N, 1)
        self.rnn_states[t + 1] = rnn_states.view(B, N, *self.rnn_states.shape[3:]) * keep.unsqueeze(-1)
        self.rnn_states_critic[t + 1] = rnn_states_critic.view(B, N, *self.rnn_states.shape[3:]) * keep.unsqueeze(-1)
        self.actions[t] = actions.view(B, N, 1).to(torch.float32)
        self.action_log_probs[t] = action_log_probs.view(B, N, 1)
        self.value_preds[t] = value_preds.view(B, N, 1)
        self.masks[t + 1] = keep
        all_done = done.all(dim=1, keepdim=True).view(B, 1, 1)
        self.active_masks[t + 1] = torch.where(all_done, torch.ones_like(keep), keep)
        self.step = (t + 1) % self.episode_length

    def after_update(self) -> None:
        """Copy the last time step to index 0 (graph_buffer.py:253-268)."""
        for name in ("obs", "node_obs", "adj_env", "rnn_states", "rnn_states_critic", "masks", "bad_masks", "active_masks"):
            x = getattr(self, name)
            x[0].copy_(x[-1])

    def _norm_mean_std(self, value_normalizer) -> Optional[Tuple[torch.Tensor, torch.Tensor]]:
        """(mean, std) as the reference's ``value_normalizer.denormalize`` applies them (x * sqrt(var) + mean):
        ``ValueNorm.running_mean_var()`` or ``PopArt.debiased_mean_var()``, sqrt taken by torch in float32."""
        if value_normalizer is None:
            return None
        if hasattr(value_normalizer, "running_mean_var"):
            mean, var = value_normalizer.running_mean_var()
        elif hasattr(value_normalizer, "debiased_mean_var"):
            mean, var = value_normalizer.debiased_mean_var()
        else:
            raise TypeError("value_normalizer: expected the reference's ValueNorm (running_mean_var) or PopArt (debiased_mean_var)")
        if mean.numel() != 1 or var.numel() != 1 or mean.dtype != torch.float32 or var.dtype != torch.float32:
            raise ValueError("value_normalizer: a float32 normaliser of one value (input_shape 1) is expected")
        mean, var = mean.detach().reshape(1), var.detach().reshape(1)
        return mean.to(self.device), torch.sqrt(var).to(self.device)

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.obs.device).cuda_stream

    def compute_returns(self, next_value: torch.Tensor, value_normalizer=None) -> None:
        """``GraphReplayBuffer.compute_returns`` (graph_buffer.py:285-366), every branch: GAE or discounted returns, with
        or without ``use_proper_time_limits``, with or without a value normaliser (the reference's ValueNorm or PopArt:
        the critic's values are then normalised and are denormalised here).  On a CUDA buffer this is one launch of
        ``fm_buffer_returns``, bit for bit the reference's float32 loop; on a CPU buffer the torch loop below."""
        norm = self._norm_mean_std(value_normalizer)
        if self.obs.is_cuda:
            import ctypes as C
            from fair_marl_b200 import _lib
            B, N = self.n_rollout_threads, self.num_agents
            c = _lib.FmReturnsConfig(episode_length=self.episode_length, num_envs=B, num_agents=N, use_gae=int(self._use_gae),
                                     use_proper_time_limits=int(self._use_proper_time_limits), gamma=float(self.gamma),
                                     gamma_lambda=float(self.gamma * self.gae_lambda))
            nv = next_value.detach().reshape(B * N).to(device=self.obs.device, dtype=torch.float32).contiguous()
            _lib.check(_lib.load().fm_buffer_returns(
                self.obs.device.index, C.byref(c), nv.data_ptr(), self.value_preds.data_ptr(), self.rewards.data_ptr(),
                self.masks.data_ptr(), self.bad_masks.data_ptr(), norm[0].data_ptr() if norm else None,
                norm[1].data_ptr() if norm else None, self.returns.data_ptr(), self._stream()), "fm_buffer_returns")
            return
        dv = (lambda x: x) if norm is None else (lambda x: x * norm[1] + norm[0])
        T = self.episode_length
        if self._use_gae:
            self.value_preds[-1] = next_value.view_as(self.value_preds[-1])
            gae = torch.zeros_like(self.value_preds[0])
            for t in reversed(range(T)):
                delta = self.rewards[t] + self.gamma * dv(self.value_preds[t + 1]) * self.masks[t + 1] - dv(self.value_preds[t])
                gae = delta + self.gamma * self.gae_lambda * self.masks[t + 1] * gae
                if self._use_proper_time_limits:
                    gae = gae * self.bad_masks[t + 1]
                self.returns[t] = gae + dv(self.value_preds[t])
        else:
            self.returns[-1] = next_value.view_as(self.returns[-1])
            for t in reversed(range(T)):
                if self._use_proper_time_limits:     # the reference denormalises in this branch only
                    self.returns[t] = ((self.returns[t + 1] * self.gamma * self.masks[t + 1] + self.rewards[t]) * self.bad_masks[t + 1]
                                       + (1 - self.bad_masks[t + 1]) * dv(self.value_preds[t]))
                else:
                    self.returns[t] = self.returns[t + 1] * self.gamma * self.masks[t + 1] + self.rewards[t]

    # ---- the trainer's input (GR_MAPPO.train, graph_mappo.py:280-359) --------------------------------------------
    def _require_cuda(self, what: str) -> None:
        if not self.obs.is_cuda:
            raise ValueError(f"DeviceRolloutBuffer.{what}: needs a CUDA buffer (fm_buffer.cu has no CPU path)")

    def advantages(self, value_normalizer=None) -> torch.Tensor:
        """The normalised advantages GR_MAPPO.train hands to the generators, [T, B, N, 1]: returns[:T] minus the
        (denormalised) values, then (adv - mean) / (std + 1e-5) with the mean and population std over the entries whose
        active_masks[:T] != 0 (np.nanmean / np.nanstd there; NaN when no entry is active).  Two launches of
        ``fm_buffer_advantages``; the (mean, std) used are left in ``advantage_stats``."""
        self._require_cuda("advantages")
        from fair_marl_b200 import _lib
        norm = self._norm_mean_std(value_normalizer)
        T, B, N = self.episode_length, self.n_rollout_threads, self.num_agents
        f32 = dict(dtype=torch.float32, device=self.obs.device)
        adv = torch.empty((T, B, N, 1), **f32)
        stats = torch.empty(2, **f32)
        ws = torch.empty(_lib.ADV_WORKSPACE_DOUBLES, dtype=torch.float64, device=self.obs.device)
        _lib.check(_lib.load().fm_buffer_advantages(
            self.obs.device.index, T, B, N, self.returns.data_ptr(), self.value_preds.data_ptr(), self.active_masks.data_ptr(),
            norm[0].data_ptr() if norm else None, norm[1].data_ptr() if norm else None, adv.data_ptr(), stats.data_ptr(),
            ws.data_ptr(), self._stream()), "fm_buffer_advantages")
        self.advantage_stats = stats
        return adv

    def feed_forward_generator(self, advantages: torch.Tensor, num_mini_batch: Optional[int] = None,
                               mini_batch_size: Optional[int] = None, generator: Optional[torch.Generator] = None):
        """``GraphReplayBuffer.feed_forward_generator``: num_mini_batch mini-batches of mini_batch_size (default
        T B N // num_mini_batch) samples drawn without replacement over (t, b, n); the remainder is dropped."""
        if num_mini_batch is None:
            raise ValueError("feed_forward_generator: num_mini_batch is required (the reference slices range(num_mini_batch))")
        return self._minibatches(advantages, "feed_forward", num_mini_batch, mini_batch_size or 0, 0, generator)

    def recurrent_generator(self, advantages: torch.Tensor, num_mini_batch: int, data_chunk_length: int,
                            generator: Optional[torch.Generator] = None):
        """``GraphReplayBuffer.recurrent_generator``: chunks of data_chunk_length consecutive steps of one (env, agent)
        column (flat over (b, n, t), so a chunk runs on into the next column when T % L != 0, as in the reference),
        num_mini_batch mini-batches of chunks // num_mini_batch chunks, rows ordered [L, chunks]; rnn states at each
        chunk's first step."""
        return self._minibatches(advantages, "recurrent", num_mini_batch, 0, data_chunk_length, generator)

    def naive_recurrent_generator(self, advantages: torch.Tensor, num_mini_batch: int,
                                  generator: Optional[torch.Generator] = None):
        """``GraphReplayBuffer.naive_recurrent_generator``: whole columns, B N // num_mini_batch per mini-batch (B N must
        be divisible by num_mini_batch), rows ordered [T, columns]; rnn states at t = 0."""
        return self._minibatches(advantages, "naive_recurrent", num_mini_batch, 0, 0, generator)

    def _minibatches(self, advantages, mode, num_mini_batch, mini_batch_size, L, generator):
        """Checks the arguments as ``fm_buffer_minibatch`` does (so a refusal raises here, before the epoch starts),
        draws the epoch's permutation on the device and returns the generator of 16-tuples."""
        self._require_cuda(mode + "_generator")
        T, B, N = self.episode_length, self.n_rollout_threads, self.num_agents
        if tuple(advantages.shape) != (T, B, N, 1) or advantages.dtype != torch.float32 or advantages.device != self.obs.device:
            raise ValueError(f"advantages: float32 [{T}, {B}, {N}, 1] on {self.obs.device} expected")
        K = int(num_mini_batch)
        if mode == "feed_forward":
            units = T * B * N
            if mini_batch_size < 0 or mini_batch_size * K > units:
                raise ValueError(f"feed_forward_generator: {K} mini-batches of {mini_batch_size} samples from {units}")
        elif mode == "recurrent":
            if L < 1:
                raise ValueError(f"recurrent_generator: data_chunk_length {L} (>= 1)")
            units = T * B * N // L
        else:
            units = B * N
        if K < 1 or K > units:
            raise ValueError(f"{mode}_generator: num_mini_batch {K} for {units} {dict(feed_forward='samples', recurrent='chunks', naive_recurrent='columns')[mode]}")
        if mode == "naive_recurrent" and units % K:
            raise ValueError(f"naive_recurrent_generator: {units} columns are not divisible by num_mini_batch {K} "
                             "(the reference would yield another number of mini-batches or raise IndexError part-way through the epoch)")
        if T * B * N >= 1 << 31:
            raise ValueError(f"{mode}_generator: T * B * N = {T * B * N} samples (at most 2^31 - 1)")
        per = mini_batch_size or units // K
        rows = per * {"feed_forward": 1, "recurrent": L, "naive_recurrent": T}[mode]
        perm = torch.randperm(units, device=self.obs.device, generator=generator)
        return self._gather_epoch(advantages.contiguous(), perm, mode, K, mini_batch_size, L, per, rows)

    def _gather_epoch(self, advantages, perm, mode, K, mini_batch_size, L, per, rows):
        import ctypes as C
        from fair_marl_b200 import _lib
        T, B, N, E = self.episode_length, self.n_rollout_threads, self.num_agents, self.num_entities
        D, F, A = self.obs.shape[-1], self.node_obs.shape[-1], self.available_actions.shape[-1]
        rnn_shape = self.rnn_states.shape[3:]
        c = _lib.FmMinibatchConfig(episode_length=T, num_envs=B, num_agents=N, num_entities=E, obs_dim=D, node_feat_dim=F,
                                   rnn_floats=rnn_shape.numel(), mode=_lib.MINIBATCH_MODES[mode], num_mini_batch=K,
                                   mini_batch_size=mini_batch_size, data_chunk_length=L)
        src = {"obs": self.obs, "node_obs": self.node_obs, "adj_env": self.adj_env, "rnn_states": self.rnn_states,
               "rnn_states_critic": self.rnn_states_critic, "actions": self.actions, "action_log_probs": self.action_log_probs,
               "value_preds": self.value_preds, "returns": self.returns, "masks": self.masks,
               "active_masks": self.active_masks, "advantages": advantages}
        slabs = _lib.FmBufferSlabs(**{k: v.data_ptr() for k, v in src.items()})
        dev = self.obs.device
        f32, i32 = dict(dtype=torch.float32, device=dev), dict(dtype=torch.int32, device=dev)
        available = self.available_actions[0, 0, :1].expand(rows, A)
        for k in range(K):
            out = {"share_obs": torch.empty((rows, N * D), **f32), "obs": torch.empty((rows, D), **f32),
                   "node_obs": torch.empty((rows, E, F), **f32), "adj": torch.empty((rows, E, E), **f32),
                   "agent_id": torch.empty((rows, 1), **i32), "share_agent_id": torch.empty((rows, N), **i32),
                   "rnn_states": torch.empty((per, *rnn_shape), **f32), "rnn_states_critic": torch.empty((per, *rnn_shape), **f32)}
            out.update({name: torch.empty((rows, 1), **f32) for name in
                        ("actions", "value_preds", "returns", "masks", "active_masks", "old_action_log_probs", "adv_targ")})
            c.mini_batch = k
            mb = _lib.FmMinibatch(**{name: t.data_ptr() for name, t in out.items()})
            _lib.check(_lib.load().fm_buffer_minibatch(dev.index, C.byref(c), C.byref(slabs), perm.data_ptr(), C.byref(mb),
                                                       self._stream()), "fm_buffer_minibatch")
            yield tuple(out[name] for name in _lib.MINIBATCH_FIELDS) + (available,)


class RolloutCollector:
    """The step loop of ``GMPERunner.run`` (graph_mpe_runner.py:60-80) with everything on the device:
    ``collect`` (policy forward on slab t) -> simulator step writing slab t + 1 -> ``insert``.  ``env`` is a
    ``B200GraphVecEnv`` or a ``B200FormationVecEnv``; the actor's ``obs_dim`` / ``node_feat_dim`` must be what it emits.

    ``max_graphs`` bounds the number of graphs per policy forward (the dense EmbedConv materialises
    ``[graphs, E, E, hidden]`` activations)."""

    def __init__(self, env, actor, critic, buffer: Optional[DeviceRolloutBuffer] = None, deterministic: bool = False,
                 max_graphs: int = 1 << 17, generator: Optional[torch.Generator] = None, fused: Optional[bool] = None,
                 **buffer_kw):
        self.env, self.actor, self.critic = env, actor, critic
        cfg = actor.cfg
        emits = (env.observation_space[0].shape[0], env.node_observation_space[0].shape[-1])
        if (cfg.obs_dim, cfg.node_feat_dim) != emits:
            raise ValueError(f"RolloutCollector: the actor takes obs_dim {cfg.obs_dim} / node_feat_dim {cfg.node_feat_dim}, the env "
                             f"emits {emits[0]} / {emits[1]} (e.g. PolicyConfig(obs_dim=11, node_feat_dim=13) for the formation family)")
        if buffer is None:
            buffer = DeviceRolloutBuffer(env.cfg.episode_length, env.num_envs, env.num_agents, env.num_entities,
                                         obs_dim=cfg.obs_dim, node_feat_dim=cfg.node_feat_dim, hidden_size=cfg.hidden_size,
                                         recurrent_N=cfg.recurrent_N, action_dim=cfg.action_dim, device=env.device, **buffer_kw)
        self.buffer = buffer
        self.deterministic, self.max_graphs, self.generator = deterministic, int(max_graphs), generator
        self._graph = None
        # fused CUDA graph network (csrc/fm_policy.cu) when both bases are in its shape family; else the dense torch modules
        from fair_marl_b200.policy import fused_gnn_supported
        E = env.num_entities
        self.fused = bool(fused) if fused is not None else (
            env.device.type == "cuda" and fused_gnn_supported(actor.cfg, E, actor.gnn_base.graph_aggr)
            and fused_gnn_supported(critic.cfg, E, critic.gnn_base.graph_aggr))

    def _critic_inputs(self, t: int, lo: int, hi: int):
        """What GMPERunner.collect feeds GR_Critic for rows lo:hi of slab t (graph_mpe_runner.py:396-436): share_obs
        (use_cent_obs) and share_agent_id (critic_graph_aggr='node', else agent_id) -> (cent_obs, agent_id, cent_env).
        The fused critic reads share_obs as the env-level slab (cent_env, no per-row copy); the dense one gets rows."""
        b, ccfg = self.buffer, self.critic.cfg
        N = b.num_agents
        if ccfg.critic_graph_aggr == "node":
            aid = b.share_agent_id[t][lo // N:hi // N].reshape(hi - lo, N)
        else:
            aid = b.agent_id[t][lo // N:hi // N].reshape(hi - lo, 1)
        cent_obs = cent_env = None
        if ccfg.use_cent_obs:
            if self.fused:
                cent_env = (b.obs[t][lo // N:hi // N].reshape(-1, N * b.obs.shape[-1]), N)
            else:
                cent_obs = b.share_obs[t][lo // N:hi // N].reshape(hi - lo, -1)
        return cent_obs, aid, cent_env

    def warmup(self) -> None:
        """``GMPERunner.warmup`` (:178-203): reset the envs; the observation lands in slab 0."""
        self.env.reset_tensor(out=self.buffer.env_views(0, with_step=False))
        self.buffer.step = 0

    @torch.no_grad()
    def collect(self, t: int) -> Tuple[torch.Tensor, ...]:
        """``GMPERunner.collect`` (:396-436) on slab ``t`` -> (values, actions, action_log_probs, rnn_states,
        rnn_states_critic), flat over (env, agent) like ``np.concatenate(buffer.x[step])``."""
        b = self.buffer
        B, N, E = b.n_rollout_threads, b.num_agents, b.num_entities
        M = B * N
        obs, node = b.obs[t].view(M, -1), b.node_obs[t].view(M, E, -1)
        adj = b.adj_env[t].unsqueeze(1).expand(B, N, E, E)
        aid = b.agent_id[t].reshape(M, 1)
        rnn, rnn_c = b.rnn_states[t].view(M, *b.rnn_states.shape[3:]), b.rnn_states_critic[t].view(M, *b.rnn_states.shape[3:])
        masks = b.masks[t].view(M, 1)
        outs = []
        per = M if self.fused else max(N, (self.max_graphs // N) * N)    # the fused kernels materialise nothing per edge: one launch
        for lo in range(0, M, per):
            hi = min(M, lo + per)
            adj_c = adj[lo // N:hi // N].reshape(hi - lo, E, E) if not self.fused else None   # stride-0 view materialised only for the torch path
            adj_e = (b.adj_env[t][lo // N:hi // N], N) if self.fused else None               # fused graph network: adj once per env
            a, lp, h = self.actor(obs[lo:hi], node[lo:hi], adj_c, aid[lo:hi], rnn[lo:hi], masks[lo:hi],
                                  deterministic=self.deterministic, generator=self.generator, adj_env=adj_e)
            cent, aid_c, cent_e = self._critic_inputs(t, lo, hi)
            v, hc = self.critic(cent, node[lo:hi], adj_c, aid_c, rnn_c[lo:hi], masks[lo:hi], adj_env=adj_e, cent_env=cent_e)
            outs.append((v, a, lp, h, hc))
        if len(outs) == 1:
            return outs[0]
        return tuple(torch.cat([o[k] for o in outs], dim=0) for k in range(5))

    @torch.no_grad()
    def _run_eager(self, steps: int) -> None:
        b = self.buffer
        B, N = b.n_rollout_threads, b.num_agents
        for _ in range(steps):
            t = b.step
            values, actions, logp, rnn, rnn_c = self.collect(t)
            a_env = b.actions_env[t]
            a_env.copy_(actions.view(B, N))
            self.env.step_tensor(a_env, out=b.env_views(t + 1))
            b.insert_policy(rnn, rnn_c, actions, logp, values)

    def run(self, steps: Optional[int] = None) -> None:
        """Collect ``steps`` (default: one episode_length) transitions into the buffer.  No host synchronisation.
        A full episode from slab 0 replays the captured CUDA graph when there is one (``capture()``)."""
        b = self.buffer
        if steps is None and b.step == 0 and self._graph is not None:
            self._graph.replay()
            return
        self._run_eager(b.episode_length if steps is None else steps)

    def capture(self) -> None:
        """Capture one episode of the loop (T x [actor + critic forward, simulator step, insert]; a few hundred small
        kernels per step) into ONE CUDA graph: at small env batches the loop is bound by launch latency, and every
        shape and pointer in it is static -- the dense policy has no data-dependent shapes and the step kernel writes
        fixed buffer slabs.  Call after at least one eager ``run()`` (library handles and the allocator are warm)."""
        b = self.buffer
        if b.step != 0:
            raise RuntimeError("capture() needs the buffer at step 0 (call after_update() after a full run())")
        dev = b.device
        g = torch.cuda.CUDAGraph()
        if self.generator is not None:
            g.register_generator_state(self.generator)
        torch.cuda.synchronize(dev)
        with torch.cuda.graph(g):
            self._run_eager(b.episode_length)
        self._graph = g                              # the capture itself does not execute: b.step is back at 0, slabs untouched

    @torch.no_grad()
    def finish(self, value_normalizer=None) -> None:
        """``GMPERunner.compute`` (:490-506): bootstrap value of the last slab, then the returns.  Pass the trainer's
        ``value_normalizer`` (ValueNorm / PopArt) when the critic is trained on normalised values (use_valuenorm, the
        reference's default): the returns are then computed from the denormalised values, as the reference does."""
        b = self.buffer
        B, N, E = b.n_rollout_threads, b.num_agents, b.num_entities
        M = B * N
        adj = b.adj_env[-1].unsqueeze(1).expand(B, N, E, E).reshape(M, E, E)
        cent, aid, cent_e = self._critic_inputs(b.episode_length, 0, M)
        v, _ = self.critic(cent, b.node_obs[-1].view(M, E, -1), adj, aid,
                           b.rnn_states_critic[-1].view(M, *b.rnn_states.shape[3:]), b.masks[-1].view(M, 1),
                           adj_env=(b.adj_env[-1], N) if self.fused else None, cent_env=cent_e)
        b.compute_returns(v, value_normalizer)
