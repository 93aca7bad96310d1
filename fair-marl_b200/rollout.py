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
                 gamma: float = 0.99, gae_lambda: float = 0.95, use_gae: bool = True, device: Any = "cuda"):
        T, B, N, E = int(episode_length), int(num_envs), int(num_agents), int(num_entities)
        self.episode_length, self.n_rollout_threads, self.num_agents, self.num_entities = T, B, N, E
        self.gamma, self.gae_lambda, self._use_gae = gamma, gae_lambda, use_gae
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

    def compute_returns(self, next_value: torch.Tensor) -> None:
        """GAE / discounted returns without value normalisation and without proper time limits
        (graph_buffer.py:314-341, the ``else`` branches)."""
        T = self.episode_length
        if self._use_gae:
            self.value_preds[-1] = next_value.view_as(self.value_preds[-1])
            gae = torch.zeros_like(self.value_preds[0])
            for t in reversed(range(T)):
                delta = self.rewards[t] + self.gamma * self.value_preds[t + 1] * self.masks[t + 1] - self.value_preds[t]
                gae = delta + self.gamma * self.gae_lambda * self.masks[t + 1] * gae
                self.returns[t] = gae + self.value_preds[t]
        else:
            self.returns[-1] = next_value.view_as(self.returns[-1])
            for t in reversed(range(T)):
                self.returns[t] = self.returns[t + 1] * self.gamma * self.masks[t + 1] + self.rewards[t]


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
    def finish(self) -> None:
        """``GMPERunner.compute`` (:490-506): bootstrap value of the last slab, then the returns."""
        b = self.buffer
        B, N, E = b.n_rollout_threads, b.num_agents, b.num_entities
        M = B * N
        adj = b.adj_env[-1].unsqueeze(1).expand(B, N, E, E).reshape(M, E, E)
        cent, aid, cent_e = self._critic_inputs(b.episode_length, 0, M)
        v, _ = self.critic(cent, b.node_obs[-1].view(M, E, -1), adj, aid,
                           b.rnn_states_critic[-1].view(M, *b.rnn_states.shape[3:]), b.masks[-1].view(M, 1),
                           adj_env=(b.adj_env[-1], N) if self.fused else None, cent_env=cent_e)
        b.compute_returns(v)
