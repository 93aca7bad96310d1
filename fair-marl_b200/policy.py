"""Dense, torch_geometric-free restatement of the reference's graph policy for the rollout loop (SURVEY.md N2).

Replaces, for the *forward* pass the rollout needs (``GMPERunner.collect``, graph_mpe_runner.py:396-436):

* ``GNNBase`` / ``TransformerConvNet`` / ``EmbedConv`` (onpolicy/algorithms/utils/gnn_new.py:23-141, :143-575;
  legacy key layout gnn.py:22-135 -- the layout of the shipped ``model_weights/*/actor.pt``),
* ``GR_Actor`` / ``GR_Critic`` (onpolicy/algorithms/graph_actor_critic.py:35-178, :258-397) with ``MLPBase``
  (utils/mlp.py), ``RNNLayer`` single-step path (utils/rnn.py:23-28) and the ``Categorical`` head (utils/act.py,
  utils/distributions.py:14-28).

The reference turns every ``[E, E]`` distance matrix into an edge list (``process_adj``, gnn_new.py:381-413),
batches the graphs through torch_geometric and scatters messages.  The graphs here are tiny (E <= 35) and all
have the same node count, so the same arithmetic is done densely on ``[graphs, E, E]`` tensors with the edge mask
``(d < max_edge_dist) & (d > 0)``: no ``nonzero`` (no host sync, no data-dependent shapes -> CUDA-graph friendly),
no index arithmetic, and the adjacency of an env is read once for its N agents.  Edge (r -> c) exists iff
``mask[r, c]``; messages flow from the row (source) to the column (target), as PyG's ``edge_index[0] -> [1]``.

This is plain PyTorch by design (BASELINE config 5: "GNN policy forward in torch"); the simulator kernels are
the product, the policy is the consumer that closes the loop on the device.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, fields
from typing import Any, Dict, Optional, Tuple

import torch
from torch import Tensor, nn


@dataclass
class PolicyConfig:
    """The fields of the reference's ``all_args`` the actor / critic read (onpolicy/config.py:264-293, :391-441)."""
    obs_dim: int = 7
    node_feat_dim: int = 11            # incl. the trailing entity-type column (gnn_new.py:129-130)
    num_agents: int = 3
    action_dim: int = 5
    num_embeddings: int = 4
    embedding_size: int = 2
    embed_hidden_size: int = 16
    embed_layer_N: int = 1
    embed_use_ReLU: bool = True
    use_feature_normalization: bool = True
    gnn_hidden_size: int = 16
    gnn_num_heads: int = 3
    gnn_concat_heads: bool = False
    gnn_layer_N: int = 2
    gnn_use_ReLU: bool = True
    max_edge_dist: float = 1.0
    hidden_size: int = 64
    layer_N: int = 1
    use_ReLU: bool = True
    use_recurrent_policy: bool = True
    use_naive_recurrent_policy: bool = False
    recurrent_N: int = 1
    actor_graph_aggr: str = "node"
    critic_graph_aggr: str = "global"
    global_aggr_type: str = "mean"
    use_cent_obs: bool = False

    @classmethod
    def from_args(cls, args: Any, **overrides) -> "PolicyConfig":
        kw = {f.name: getattr(args, f.name) for f in fields(cls) if hasattr(args, f.name)}
        kw.update(overrides)
        return cls(**kw)

    @property
    def gnn_out_dim(self) -> int:
        return self.gnn_hidden_size * (self.gnn_num_heads if self.gnn_concat_heads else 1)


def edge_mask(adj: Tensor, max_edge_dist: float) -> Tensor:
    """``process_adj``'s connectivity (gnn_new.py:392): strict ``<`` and ``> 0``.  bool, same shape as ``adj``."""
    return (adj < max_edge_dist) & (adj > 0)


def _act(relu: bool) -> nn.Module:
    return nn.ReLU() if relu else nn.Tanh()


def _norm_rows(norm: nn.Module, h: Tensor) -> Tensor:
    """LayerNorm over a short last dimension of a large tensor (the [graphs, E, E, 16] edge messages).  torch's native
    kernel spends one thread block per 16-element row, and its row reductions (var_mean) run at a fraction of the
    memory bandwidth; here the two row statistics are thin GEMMs against a constant vector (rows x C @ C x 1, which
    stream the tensor once at full bandwidth) and the rest is elementwise.  Same formula: two-pass mean / biased
    variance of the centred values, eps inside the root."""
    if not isinstance(norm, nn.LayerNorm):
        return norm(h)
    C = h.shape[-1]
    ones = torch.full((C, 1), 1.0 / C, dtype=h.dtype, device=h.device)
    flat = h.reshape(-1, C)
    centred = flat - flat @ ones
    var = (centred * centred) @ ones
    out = centred * torch.rsqrt(var + norm.eps)
    return torch.addcmul(norm.bias, out, norm.weight).view(h.shape)


class DenseEmbedConv(nn.Module):
    """``EmbedConv`` (gnn_new.py:23-141): message of edge (r -> c) =
    MLP([x_r[:-1], embed(type_r), d_rc]), summed over the incoming edges of c.

    The first linear layer splits into a per-node part and a rank-1 per-edge part,
    ``W [x_r, emb_r, d_rc] + b = (W_n [x_r, emb_r] + b) + w_d d_rc``, so the node part is computed once per node
    rather than once per edge.  LayerNorms are one module per position; the gnn_new layout shares a single
    LayerNorm between all of them (gnn_new.py:67, :94) and ``load_reference_state_dict`` copies it into each.
    """

    def __init__(self, cfg: PolicyConfig):
        super().__init__()
        H = cfg.embed_hidden_size
        self.entity_embed = nn.Embedding(cfg.num_embeddings, cfg.embedding_size)
        self.lin1 = nn.Linear(cfg.node_feat_dim - 1 + cfg.embedding_size + 1, H)
        self.act = _act(cfg.embed_use_ReLU)
        ln = (lambda: nn.LayerNorm(H)) if cfg.use_feature_normalization else (lambda: nn.Identity())
        self.norm1 = ln()
        self.hidden = nn.ModuleList([nn.Linear(H, H) for _ in range(cfg.embed_layer_N)])
        self.hidden_norm = nn.ModuleList([ln() for _ in range(cfg.embed_layer_N)])

    def forward(self, x: Tensor, adj: Tensor, mask: Tensor) -> Tensor:
        # x [M, E, F], adj / mask [M, E(row = source), E(col = target)]
        feat, typ = x[..., :-1], x[..., -1].long()
        node_in = torch.cat([feat, self.entity_embed(typ)], dim=-1)
        W = self.lin1.weight
        h_node = torch.nn.functional.linear(node_in, W[:, :-1], self.lin1.bias)          # [M, E, H]
        h = torch.addcmul(h_node.unsqueeze(2), adj.unsqueeze(-1), W[:, -1])             # [M, E_r, E_c, H], one pass
        h = _norm_rows(self.norm1, self.act(h))
        for lin, norm in zip(self.hidden, self.hidden_norm):
            h = _norm_rows(norm, self.act(lin(h)))
        return (h * mask.unsqueeze(-1).to(h.dtype)).sum(dim=1)                          # sum over sources r -> [M, E_c, H]


class DenseTransformerConv(nn.Module):
    """PyG ``TransformerConv(heads, concat, beta=False, edge_dim=1, root_weight=True)`` on dense graphs
    (constructed at gnn_new.py:252-271).  With a scalar edge attribute d the edge projection is rank 1,
    ``W_e d = d w_e``, so  q_t . (k_s + d_st w_e) = q_t . k_s + d_st (q_t . w_e)  and
    sum_s alpha_ts (v_s + d_st w_e) = alpha @ v + (sum_s alpha_ts d_st) w_e."""

    def __init__(self, in_channels: int, out_channels: int, heads: int, concat: bool):
        super().__init__()
        self.heads, self.out_channels, self.concat = heads, out_channels, concat
        HC = heads * out_channels
        self.lin_key = nn.Linear(in_channels, HC)
        self.lin_query = nn.Linear(in_channels, HC)
        self.lin_value = nn.Linear(in_channels, HC)
        self.lin_edge = nn.Linear(1, HC, bias=False)
        self.lin_skip = nn.Linear(in_channels, HC if concat else out_channels)

    def forward(self, x: Tensor, adj: Tensor, mask: Tensor) -> Tensor:
        M, E, _ = x.shape
        H, C = self.heads, self.out_channels
        q = self.lin_query(x).view(M, E, H, C).transpose(1, 2)                           # [M, H, E_t, C]
        k = self.lin_key(x).view(M, E, H, C).transpose(1, 2)                             # [M, H, E_s, C]
        v = self.lin_value(x).view(M, E, H, C).transpose(1, 2)
        we = self.lin_edge.weight.view(H, C)
        d_ts = adj.transpose(1, 2).unsqueeze(1)                                          # [M, 1, E_t, E_s] = d[s, t]
        m_ts = mask.transpose(1, 2).unsqueeze(1)
        qe = (q * we.view(1, H, 1, C)).sum(-1, keepdim=True)                             # q_t . w_e  [M, H, E_t, 1]
        score = (q @ k.transpose(-1, -2) + qe * d_ts) * (1.0 / math.sqrt(C))
        score = score.masked_fill(~m_ts, float("-inf"))
        alpha = torch.softmax(score, dim=-1)
        alpha = torch.nan_to_num(alpha, nan=0.0)                                         # targets without incoming edges
        out = alpha @ v + (alpha * d_ts).sum(-1, keepdim=True) * we.view(1, H, 1, C)     # [M, H, E_t, C]
        out = out.transpose(1, 2)
        out = out.reshape(M, E, H * C) if self.concat else out.mean(dim=2)
        return out + self.lin_skip(x)


_AGGR_CODE = {"node": 0, "mean": 1, "max": 2, "add": 3}


def fused_gnn_supported(cfg: PolicyConfig, num_entities: int, graph_aggr: str) -> bool:
    """Shape family of the fused CUDA forward (csrc/fm_policy.cu): the configuration of the shipped model_weights, at any
    graph size a fused kernel covers (``fm_gnn_mapping``: 2 <= E <= 64)."""
    from fair_marl_b200 import _lib
    ok = (cfg.embed_hidden_size == 16 and cfg.gnn_hidden_size == 16 and cfg.gnn_num_heads == 3 and not cfg.gnn_concat_heads
          and cfg.embed_layer_N <= 2 and cfg.num_embeddings <= 4 and cfg.embed_use_ReLU == cfg.gnn_use_ReLU
          and (graph_aggr == "node" or cfg.global_aggr_type in ("mean", "max", "add")))
    return bool(ok and _lib.load().fm_gnn_mapping(int(num_entities), int(cfg.node_feat_dim)) != 0)


def pack_gnn_weights(gnn: "DenseGNNBase") -> Tensor:
    """The weight blob ``fm_gnn_forward`` reads (layout: include/fairmarl.h ``FmGnnConfig``): lin1 split into its
    node-feature part (transposed, padded to 16 rows), the per-entity-type constant ``W_emb . embed(type) + b`` and the
    edge-attribute column; every later matrix transposed to [in][out]; query | key | value | skip of a conv side by side."""
    cfg, emb = gnn.cfg, gnn.embed_layer
    H, KF = cfg.embed_hidden_size, cfg.node_feat_dim - 1
    dev, dt = emb.lin1.weight.device, torch.float32
    W1 = emb.lin1.weight.detach().to(dt)                                  # [H, KF + emb + 1]
    es = cfg.embedding_size
    parts = []
    wn = torch.zeros(16, H, dtype=dt, device=dev)
    wn[:KF] = W1[:, :KF].t()
    parts.append(wn.reshape(-1))
    ty = torch.zeros(4, H, dtype=dt, device=dev)
    table = emb.entity_embed.weight.detach().to(dt)                        # [num_embeddings, es]
    ty[:table.shape[0]] = table @ W1[:, KF:KF + es].t() + emb.lin1.bias.detach().to(dt)
    parts.append(ty.reshape(-1))
    parts.append(W1[:, KF + es].contiguous())

    def ln_params(norm):
        if isinstance(norm, nn.LayerNorm):
            return [norm.weight.detach().to(dt), norm.bias.detach().to(dt)]
        return [torch.ones(H, dtype=dt, device=dev), torch.zeros(H, dtype=dt, device=dev)]

    parts += ln_params(emb.norm1)
    for lin, norm in zip(emb.hidden, emb.hidden_norm):
        parts += [lin.weight.detach().to(dt).t().reshape(-1), lin.bias.detach().to(dt)] + ln_params(norm)
    for conv in [gnn.gnn1] + list(gnn.gnn2):
        Wc = torch.cat([conv.lin_query.weight, conv.lin_key.weight, conv.lin_value.weight, conv.lin_skip.weight], dim=0).detach().to(dt)
        bc = torch.cat([conv.lin_query.bias, conv.lin_key.bias, conv.lin_value.bias, conv.lin_skip.bias]).detach().to(dt)
        parts += [Wc.t().reshape(-1), bc, conv.lin_edge.weight.detach().to(dt).reshape(-1)]
    return torch.cat([x.reshape(-1) for x in parts]).contiguous()


class DenseGNNBase(nn.Module):
    """``GNNBase.forward`` (gnn_new.py:555-575) = process_adj -> EmbedConv -> act(TransformerConv) x (1 + layer_N)
    -> node gather (``graph_aggr='node'``) or global pool.

    Two implementations of the same function: ``forward`` with ``adj_env=None`` is plain PyTorch (any configuration,
    any device); with ``adj_env=(adj [B, E, E], graphs_per_adj)`` on a CUDA device and a supported configuration
    (``fused_gnn_supported``) the whole base is ONE launch of the fused kernel ``fm_gnn_forward`` (csrc/fm_policy.cu),
    which reads the adjacency once per env.  Inference only (no autograd through the fused path)."""

    def __init__(self, cfg: PolicyConfig, graph_aggr: str):
        super().__init__()
        self.cfg, self.graph_aggr = cfg, graph_aggr
        self.embed_layer = DenseEmbedConv(cfg)
        C, H = cfg.gnn_hidden_size, cfg.gnn_num_heads
        self.gnn1 = DenseTransformerConv(cfg.embed_hidden_size, C, H, cfg.gnn_concat_heads)
        nxt = C * H if cfg.gnn_concat_heads else C
        self.gnn2 = nn.ModuleList([DenseTransformerConv(nxt, C, H, cfg.gnn_concat_heads) for _ in range(cfg.gnn_layer_N)])
        self.act = _act(cfg.gnn_use_ReLU)
        self.out_dim = cfg.gnn_out_dim

    def fused_available(self, node_obs: Tensor) -> bool:
        return (node_obs.is_cuda and not torch.is_grad_enabled() and node_obs.dtype == torch.float32
                and fused_gnn_supported(self.cfg, node_obs.shape[1], self.graph_aggr))

    def _packed(self) -> Tensor:
        key = tuple((p.data_ptr(), p._version) for p in self.parameters())
        if getattr(self, "_pack_key", None) != key:
            self._pack_key, self._pack = key, pack_gnn_weights(self)
        return self._pack

    def forward_fused(self, node_obs: Tensor, adj_env: Tensor, graphs_per_adj: int, agent_id: Optional[Tensor],
                      mapping: int = 0) -> Tensor:
        """One launch of ``fm_gnn_forward``.  node_obs [M, E, F] contiguous fp32; adj_env [M / graphs_per_adj, E, E];
        agent_id [M] or [M, 1] node indices (aggr 'node'), or [M, k] with k > 1: the k nodes' features side by side
        ([M, k * 16], ``fm_gnn_gather``).  ``mapping``: 0 auto, 1 the warp-per-graph kernel, 2 the CTA-per-graph kernel
        (``FmGnnConfig.mapping``)."""
        import ctypes as C
        from fair_marl_b200 import _lib
        cfg = self.cfg
        M, E, F = node_obs.shape
        if not node_obs.is_contiguous() or not adj_env.is_contiguous() or adj_env.shape[0] * graphs_per_adj != M:
            raise ValueError("forward_fused: node_obs / adj_env must be contiguous and adj_env.shape[0] * graphs_per_adj == M")
        aggr = 0 if self.graph_aggr == "node" else _AGGR_CODE[cfg.global_aggr_type]
        c = _lib.FmGnnConfig(num_graphs=M, graphs_per_adj=int(graphs_per_adj), num_entities=E, node_feat_dim=F,
                             embed_layers=cfg.embed_layer_N, conv_layers=1 + cfg.gnn_layer_N, aggr=aggr,
                             relu=int(cfg.gnn_use_ReLU), layer_norm=int(cfg.use_feature_normalization),
                             mapping=int(mapping), max_edge_dist=float(cfg.max_edge_dist))
        w = self._packed()
        aid = None
        stream = torch.cuda.current_stream(node_obs.device).cuda_stream
        if aggr == 0:
            if agent_id is None or agent_id.numel() == 0 or agent_id.numel() % max(M, 1) != 0:
                raise ValueError("forward_fused: aggr 'node' gathers k nodes per graph (agent_id [M] or [M, k])")
            k = agent_id.numel() // max(M, 1)
            if k > 1:
                aid = agent_id.reshape(M, k).to(torch.int32).contiguous()
                out = torch.empty((M, k * cfg.gnn_hidden_size), dtype=torch.float32, device=node_obs.device)
                _lib.check(_lib.load().fm_gnn_gather(node_obs.device.index, C.byref(c), k, w.data_ptr(), node_obs.data_ptr(),
                                                     adj_env.data_ptr(), aid.data_ptr(), out.data_ptr(), stream), "fm_gnn_gather")
                return out
            aid = agent_id.reshape(M).to(torch.int32).contiguous()
        out = torch.empty((M, cfg.gnn_hidden_size), dtype=torch.float32, device=node_obs.device)
        _lib.check(_lib.load().fm_gnn_forward(node_obs.device.index, C.byref(c), w.data_ptr(), node_obs.data_ptr(),
                                              adj_env.data_ptr(), aid.data_ptr() if aid is not None else None,
                                              out.data_ptr(), stream), "fm_gnn_forward")
        return out

    def forward(self, node_obs: Tensor, adj: Tensor, agent_id: Tensor, adj_env: Optional[Tuple[Tensor, int]] = None) -> Tensor:
        """node_obs [M, E, F]; adj [M, E, E] (any stride, e.g. the env's matrix expanded over its agents);
        agent_id [M, k] integer node indices.  ``adj_env``: see the class docstring."""
        if adj_env is not None and self.fused_available(node_obs):
            return self.forward_fused(node_obs.contiguous(), adj_env[0], adj_env[1], agent_id)
        mask = edge_mask(adj, self.cfg.max_edge_dist)
        x = self.embed_layer(node_obs, adj, mask)
        x = self.act(self.gnn1(x, adj, mask))
        for g in self.gnn2:
            x = self.act(g(x, adj, mask))
        if self.graph_aggr == "node":
            idx = agent_id.long().unsqueeze(-1).expand(-1, -1, x.size(-1))
            return x.gather(1, idx).flatten(1)
        how = self.cfg.global_aggr_type
        if how == "mean":
            return x.mean(dim=1)
        if how == "max":
            return x.max(dim=1).values
        if how == "add":
            return x.sum(dim=1)
        raise ValueError(f"Invalid global_aggr_type: {how}")


class _MLPBase(nn.Module):
    """``MLPBase`` (utils/mlp.py): LayerNorm(in) -> [Linear, act, LayerNorm] x (1 + layer_N)."""

    def __init__(self, cfg: PolicyConfig, in_dim: int):
        super().__init__()
        self.feature_norm = nn.LayerNorm(in_dim) if cfg.use_feature_normalization else nn.Identity()
        dims = [in_dim] + [cfg.hidden_size] * (1 + cfg.layer_N)
        self.lins = nn.ModuleList([nn.Linear(a, b) for a, b in zip(dims[:-1], dims[1:])])
        self.norms = nn.ModuleList([nn.LayerNorm(cfg.hidden_size) for _ in range(1 + cfg.layer_N)])
        self.act = _act(cfg.use_ReLU)

    def forward(self, x: Tensor) -> Tensor:
        x = self.feature_norm(x)
        for lin, norm in zip(self.lins, self.norms):
            x = norm(self.act(lin(x)))
        return x


class _RNNStep(nn.Module):
    """``RNNLayer`` for one time step (utils/rnn.py:23-28, :57): GRU on ``h * mask``, then LayerNorm."""

    def __init__(self, cfg: PolicyConfig):
        super().__init__()
        self.recurrent_N = cfg.recurrent_N
        self.rnn = nn.GRU(cfg.hidden_size, cfg.hidden_size, num_layers=cfg.recurrent_N)
        self.norm = nn.LayerNorm(cfg.hidden_size)

    def forward(self, x: Tensor, hxs: Tensor, masks: Tensor) -> Tuple[Tensor, Tensor]:
        # One GRU step per layer written out (torch.nn.GRU's equations on its own parameters): two fp32 GEMMs per
        # layer instead of a cuDNN sequence call of length 1 (which would also switch to TF32 by default).
        h_in = hxs * masks.view(-1, 1, 1)                                   # [M, recurrent_N, H]
        outs = []
        for layer in range(self.recurrent_N):
            w_ih, w_hh = getattr(self.rnn, f"weight_ih_l{layer}"), getattr(self.rnn, f"weight_hh_l{layer}")
            b_ih, b_hh = getattr(self.rnn, f"bias_ih_l{layer}"), getattr(self.rnn, f"bias_hh_l{layer}")
            h = h_in[:, layer]
            gi = torch.nn.functional.linear(x, w_ih, b_ih)
            gh = torch.nn.functional.linear(h, w_hh, b_hh)
            i_r, i_z, i_n = gi.chunk(3, dim=1)
            h_r, h_z, h_n = gh.chunk(3, dim=1)
            r = torch.sigmoid(i_r + h_r)
            z = torch.sigmoid(i_z + h_z)
            n = torch.tanh(i_n + r * h_n)
            x = (1.0 - z) * n + z * h
            outs.append(x)
        return self.norm(x), torch.stack(outs, dim=1)


def _quad_interleave(w_t: Tensor, rows: int) -> Tensor:
    """W^T [K, C] (zero padded to ``rows`` rows) -> [rows / 4][C][4], the layout the head kernel reads with one LDS.128 per
    (k-quad, column)."""
    K, Ccols = w_t.shape
    pad = torch.zeros(rows, Ccols, dtype=w_t.dtype, device=w_t.device)
    pad[:K] = w_t
    return pad.view(rows // 4, 4, Ccols).permute(0, 2, 1).contiguous().reshape(-1)


class _Trunk(nn.Module):
    def __init__(self, cfg: PolicyConfig, graph_aggr: str, extra_in: int, gnn_mult: int = 1):
        super().__init__()
        self.cfg = cfg
        self.gnn_base = DenseGNNBase(cfg, graph_aggr)
        self.base = _MLPBase(cfg, self.gnn_base.out_dim * gnn_mult + extra_in)
        self.recurrent = cfg.use_recurrent_policy or cfg.use_naive_recurrent_policy
        if self.recurrent:
            self.rnn = _RNNStep(cfg)
        self._head_in = self.gnn_base.out_dim * gnn_mult + extra_in

    # ---- fused head (csrc/fm_policy.cu head_kernel, fm_policy_head) -------------------------------------------------
    def head_supported(self) -> bool:
        cfg = self.cfg
        return (cfg.hidden_size == 64 and cfg.layer_N <= 2 and self.gnn_base.out_dim == 16 and 16 <= self._head_in <= 32
                and (not self.recurrent or cfg.recurrent_N == 1))

    def _out_linear(self) -> nn.Linear:
        raise NotImplementedError

    def pack_head_weights(self, width: int = 32) -> Tensor:
        """The weight blob ``fm_policy_head`` reads (layout: include/fairmarl.h ``FmHeadConfig``), or with ``width`` the
        padded input width Dp of the blob ``fm_critic_head`` reads (``FmCriticHeadConfig``): the two differ only in the
        width of the feature norm and of fc1."""
        base, dt = self.base, torch.float32
        dev = base.lins[0].weight.device
        D, H = self._head_in, 64
        g, b = torch.ones(width, dtype=dt, device=dev), torch.zeros(width, dtype=dt, device=dev)
        if isinstance(base.feature_norm, nn.LayerNorm):
            g[:D], b[:D] = base.feature_norm.weight.detach().to(dt), base.feature_norm.bias.detach().to(dt)
        parts = [g, b]
        for k, (lin, norm) in enumerate(zip(base.lins, base.norms)):
            parts += [_quad_interleave(lin.weight.detach().to(dt).t(), width if k == 0 else H), lin.bias.detach().to(dt),
                      norm.weight.detach().to(dt), norm.bias.detach().to(dt)]
        if self.recurrent:
            r = self.rnn.rnn
            parts += [_quad_interleave(r.weight_ih_l0.detach().to(dt).t(), H), _quad_interleave(r.weight_hh_l0.detach().to(dt).t(), H),
                      r.bias_ih_l0.detach().to(dt), r.bias_hh_l0.detach().to(dt),
                      self.rnn.norm.weight.detach().to(dt), self.rnn.norm.bias.detach().to(dt)]
        out = self._out_linear()
        wo, bo = torch.zeros(8, H, dtype=dt, device=dev), torch.zeros(8, dtype=dt, device=dev)
        wo[:out.weight.shape[0]], bo[:out.bias.shape[0]] = out.weight.detach().to(dt), out.bias.detach().to(dt)
        parts += [wo.reshape(-1), bo]
        return torch.cat([x.reshape(-1) for x in parts]).contiguous()

    def _packed_head(self, width: int = 32) -> Tensor:
        ps = [p for n, p in self.named_parameters() if not n.startswith("gnn_base.")]
        key = (width,) + tuple((p.data_ptr(), p._version) for p in ps)
        if getattr(self, "_head_key", None) != key:
            self._head_key, self._head_pack = key, self.pack_head_weights(width)
        return self._head_pack

    def _run_head(self, obs: Optional[Tensor], nbd: Tensor, rnn_states: Tensor, masks: Tensor, u: Optional[Tensor], critic: bool):
        import ctypes as C
        from fair_marl_b200 import _lib
        cfg = self.cfg
        M = nbd.shape[0]
        out_dim = self._out_linear().weight.shape[0]
        c = _lib.FmHeadConfig(num_rows=M, obs_dim=0 if obs is None else obs.shape[1], layers=cfg.layer_N,
                              recurrent=int(self.recurrent), feature_norm=int(cfg.use_feature_normalization),
                              relu=int(cfg.use_ReLU), num_outputs=out_dim)
        dev = nbd.device
        w = self._packed_head()
        rnn_in = rnn_states.reshape(M, -1).contiguous() if self.recurrent else None
        rnn_out = torch.empty((M, 1, 64), dtype=torch.float32, device=dev) if self.recurrent else rnn_states
        mk = masks.reshape(M).to(torch.float32).contiguous() if self.recurrent else None
        ptr = lambda t: t.data_ptr() if t is not None else None
        if critic:
            value = torch.empty((M, 1), dtype=torch.float32, device=dev)
            logp = action = None
        else:
            value = None
            logp = torch.empty((M, 1), dtype=torch.float32, device=dev)
            action = torch.empty((M, 1), dtype=torch.int64, device=dev)
        if obs is not None:
            obs = obs.contiguous()
        _lib.check(_lib.load().fm_policy_head(dev.index, C.byref(c), w.data_ptr(), ptr(obs), nbd.data_ptr(), ptr(rnn_in), ptr(mk),
                                              ptr(u), ptr(rnn_out) if self.recurrent else None, ptr(logp), ptr(action), ptr(value),
                                              torch.cuda.current_stream(dev).cuda_stream), "fm_policy_head")
        return (value, rnn_out) if critic else (action, logp, rnn_out)


class DenseGraphActor(_Trunk):
    """``GR_Actor.forward`` (graph_actor_critic.py:93-178) for Discrete actions."""

    def __init__(self, cfg: PolicyConfig):
        super().__init__(cfg, cfg.actor_graph_aggr, cfg.obs_dim)
        self.action_out = nn.Linear(cfg.hidden_size, cfg.action_dim)

    def _out_linear(self) -> nn.Linear:
        return self.action_out

    def features(self, obs, node_obs, adj, agent_id, rnn_states, masks, adj_env=None):
        nbd = self.gnn_base(node_obs, adj, agent_id, adj_env=adj_env)
        x = self.base(torch.cat([obs, nbd], dim=1))
        if self.recurrent:
            x, rnn_states = self.rnn(x, rnn_states, masks)
        return x, rnn_states

    def forward(self, obs: Tensor, node_obs: Tensor, adj: Tensor, agent_id: Tensor, rnn_states: Tensor, masks: Tensor,
                available_actions: Optional[Tensor] = None, deterministic: bool = False,
                generator: Optional[torch.Generator] = None,
                adj_env: Optional[Tuple[Tensor, int]] = None) -> Tuple[Tensor, Tensor, Tensor]:
        """-> (actions [M,1] int64, action_log_probs [M,1], rnn_states [M,recurrent_N,hidden]).
        ``adj_env = (adj [B, E, E], graphs_per_adj)`` selects the fused CUDA graph network (``DenseGNNBase``) and, when the
        head is in its shape family too, the fused head kernel (``fm_policy_head``): two launches for the whole forward."""
        if (adj_env is not None and available_actions is None and self.cfg.actor_graph_aggr == "node" and self.head_supported()
                and self.cfg.action_dim <= 8 and self.gnn_base.fused_available(node_obs) and agent_id.numel() == node_obs.shape[0]):
            nbd = self.gnn_base.forward_fused(node_obs.contiguous(), adj_env[0], adj_env[1], agent_id)
            u = None if deterministic else torch.rand(nbd.shape[0], device=nbd.device, generator=generator)
            return self._run_head(obs, nbd, rnn_states, masks, u, critic=False)
        x, rnn_states = self.features(obs, node_obs, adj, agent_id, rnn_states, masks, adj_env=adj_env)
        logits = self.action_out(x)
        if available_actions is not None:                                   # distributions.py:86-88
            logits = logits.masked_fill(available_actions == 0, -1e10)
        logp = torch.log_softmax(logits, dim=-1)
        if deterministic:
            actions = logp.argmax(dim=-1, keepdim=True)                       # FixedCategorical.mode
        else:
            actions = torch.multinomial(logp.exp(), 1, generator=generator)   # FixedCategorical.sample
        return actions, logp.gather(1, actions), rnn_states


class DenseGraphCritic(_Trunk):
    """``GR_Critic.forward`` (graph_actor_critic.py:323-397); ``v_out`` is a Linear (PopArt's forward is the same
    affine map, utils/popart.py)."""

    def __init__(self, cfg: PolicyConfig):
        mult = cfg.num_agents if cfg.critic_graph_aggr == "node" else 1
        super().__init__(cfg, cfg.critic_graph_aggr, cfg.obs_dim * cfg.num_agents if cfg.use_cent_obs else 0, mult)
        self.v_out = nn.Linear(cfg.hidden_size, 1)

    def _out_linear(self) -> nn.Linear:
        return self.v_out

    # fm_critic_head's input width cap (csrc/fm_launch.h CRITIC_HEAD_MAX_IN)
    CRITIC_HEAD_MAX_IN = 768

    def critic_head_supported(self) -> bool:
        """The fused heads cover this critic: ``fm_policy_head`` for inputs of at most 32 features, ``fm_critic_head``
        above that, up to CRITIC_HEAD_MAX_IN."""
        cfg = self.cfg
        return (cfg.hidden_size == 64 and cfg.layer_N <= 2 and self.gnn_base.out_dim == 16 and self._head_in <= self.CRITIC_HEAD_MAX_IN
                and (not self.recurrent or cfg.recurrent_N == 1))

    def _run_critic_head(self, cent: Optional[Tuple[Tensor, int]], nbd: Tensor, rnn_states: Tensor, masks: Tensor):
        """One launch of ``fm_critic_head``: cent = (cent_obs [M / rows_per_env, cent_dim], rows_per_env) or None; nbd
        [M, nbd_dim] -> (values [M, 1], rnn_states)."""
        import ctypes as C
        from fair_marl_b200 import _lib
        cfg = self.cfg
        M, dev = nbd.shape[0], nbd.device
        cent_obs = cent[0].contiguous() if cent is not None else None
        c = _lib.FmCriticHeadConfig(num_rows=M, cent_dim=0 if cent is None else cent_obs.shape[1],
                                    rows_per_env=1 if cent is None else int(cent[1]), nbd_dim=nbd.shape[1], layers=cfg.layer_N,
                                    recurrent=int(self.recurrent), feature_norm=int(cfg.use_feature_normalization),
                                    relu=int(cfg.use_ReLU))
        if cent is not None and cent_obs.shape[0] * c.rows_per_env != M:
            raise ValueError("_run_critic_head: cent_obs must hold one row per rows_per_env rows")
        w = self._packed_head((self._head_in + 31) // 32 * 32)
        nbd = nbd.contiguous()
        rnn_in = rnn_states.reshape(M, -1).contiguous() if self.recurrent else None
        rnn_out = torch.empty((M, 1, 64), dtype=torch.float32, device=dev) if self.recurrent else rnn_states
        mk = masks.reshape(M).to(torch.float32).contiguous() if self.recurrent else None
        value = torch.empty((M, 1), dtype=torch.float32, device=dev)
        ptr = lambda t: t.data_ptr() if t is not None else None
        _lib.check(_lib.load().fm_critic_head(dev.index, C.byref(c), w.data_ptr(), ptr(cent_obs), nbd.data_ptr(), ptr(rnn_in),
                                              ptr(mk), ptr(rnn_out) if self.recurrent else None, value.data_ptr(),
                                              torch.cuda.current_stream(dev).cuda_stream), "fm_critic_head")
        return value, rnn_out

    def forward(self, cent_obs: Optional[Tensor], node_obs: Tensor, adj: Tensor, agent_id: Tensor, rnn_states: Tensor,
                masks: Tensor, adj_env: Optional[Tuple[Tensor, int]] = None,
                cent_env: Optional[Tuple[Tensor, int]] = None) -> Tuple[Tensor, Tensor]:
        """cent_obs [M, N * obs_dim] (use_cent_obs; ``share_obs``) or, without a per-row copy, ``cent_env =
        (obs [M / rows_per_env, N * obs_dim], rows_per_env)``: one row per env, read by its rows_per_env ego graphs, as
        ``adj_env`` passes the adjacency.  agent_id [M, 1], or [M, N] (``share_agent_id``) for critic_graph_aggr='node'.
        With ``adj_env`` and a covered configuration (``critic_head_supported``) this is two launches: the fused graph
        network (a k-node gather for 'node') and the fused head, chosen by the input width D: ``fm_policy_head`` for
        D <= 32, ``fm_critic_head`` above.  Otherwise the dense modules."""
        cent = None
        if self.cfg.use_cent_obs:
            cent = cent_env if cent_env is not None else (cent_obs, 1)
        if adj_env is not None and self.critic_head_supported() and self.gnn_base.fused_available(node_obs):
            nbd = self.gnn_base.forward_fused(node_obs.contiguous(), adj_env[0], adj_env[1],
                                              agent_id if self.cfg.critic_graph_aggr == "node" else None)
            if self._head_in > 32:
                return self._run_critic_head(cent, nbd, rnn_states, masks)
            x = nbd if cent is None else torch.cat([cent[0].repeat_interleave(cent[1], dim=0), nbd], dim=1)
            D = x.shape[1]
            return self._run_head(x[:, :D - 16] if D > 16 else None, x[:, D - 16:].contiguous(), rnn_states, masks, None, critic=True)
        nbd = self.gnn_base(node_obs, adj, agent_id, adj_env=adj_env)
        if cent is not None and cent_obs is None:
            cent_obs = cent[0].repeat_interleave(cent[1], dim=0)
        x = torch.cat([cent_obs, nbd], dim=1) if self.cfg.use_cent_obs else nbd
        x = self.base(x)
        if self.recurrent:
            x, rnn_states = self.rnn(x, rnn_states, masks)
        return self.v_out(x), rnn_states


# ------------------------------------------------------------------------------------------------------------
def _map_reference_keys(sd: Dict[str, Tensor], cfg: PolicyConfig, head: str) -> Dict[str, Tensor]:
    """Reference state-dict keys (``GR_Actor`` / ``GR_Critic``; gnn_new.py layout or the legacy gnn.py layout of the
    shipped ``model_weights``) -> keys of the dense modules above."""
    out: Dict[str, Tensor] = {}
    e = "gnn_base.gnn.embed_layer."
    legacy = (e + "lin1.0.weight") in sd
    out["gnn_base.embed_layer.entity_embed.weight"] = sd[e + "entity_embed.weight"]
    ln = cfg.use_feature_normalization
    if legacy:                                             # gnn.py:75-85: lin1 = Seq(Linear, act, LN); lin2 = clones of lin_h
        out["gnn_base.embed_layer.lin1.weight"] = sd[e + "lin1.0.weight"]
        out["gnn_base.embed_layer.lin1.bias"] = sd[e + "lin1.0.bias"]
        if ln:
            out["gnn_base.embed_layer.norm1.weight"] = sd[e + "lin1.2.weight"]
            out["gnn_base.embed_layer.norm1.bias"] = sd[e + "lin1.2.bias"]
        for i in range(cfg.embed_layer_N):
            out[f"gnn_base.embed_layer.hidden.{i}.weight"] = sd[e + f"lin2.{i}.0.weight"]
            out[f"gnn_base.embed_layer.hidden.{i}.bias"] = sd[e + f"lin2.{i}.0.bias"]
            if ln:
                out[f"gnn_base.embed_layer.hidden_norm.{i}.weight"] = sd[e + f"lin2.{i}.2.weight"]
                out[f"gnn_base.embed_layer.hidden_norm.{i}.bias"] = sd[e + f"lin2.{i}.2.bias"]
    else:                                                  # gnn_new.py:86-95: one shared LayerNorm, layers = [Linear, act, LN] * N
        out["gnn_base.embed_layer.lin1.weight"] = sd[e + "lin1.weight"]
        out["gnn_base.embed_layer.lin1.bias"] = sd[e + "lin1.bias"]
        if ln:
            out["gnn_base.embed_layer.norm1.weight"] = sd[e + "layer_norm.weight"]
            out["gnn_base.embed_layer.norm1.bias"] = sd[e + "layer_norm.bias"]
        for i in range(cfg.embed_layer_N):
            out[f"gnn_base.embed_layer.hidden.{i}.weight"] = sd[e + f"layers.{3 * i}.weight"]
            out[f"gnn_base.embed_layer.hidden.{i}.bias"] = sd[e + f"layers.{3 * i}.bias"]
            if ln:
                out[f"gnn_base.embed_layer.hidden_norm.{i}.weight"] = sd[e + "layer_norm.weight"]
                out[f"gnn_base.embed_layer.hidden_norm.{i}.bias"] = sd[e + "layer_norm.bias"]
    convs = [("gnn_base.gnn.gnn1.", "gnn_base.gnn1.")] + [(f"gnn_base.gnn.gnn2.{i}.", f"gnn_base.gnn2.{i}.")
                                                           for i in range(cfg.gnn_layer_N)]
    for src, dst in convs:
        for name in ("lin_key.weight", "lin_key.bias", "lin_query.weight", "lin_query.bias", "lin_value.weight",
                     "lin_value.bias", "lin_edge.weight", "lin_skip.weight", "lin_skip.bias"):
            out[dst + name] = sd[src + name]
    if ln:
        out["base.feature_norm.weight"] = sd["base.feature_norm.weight"]
        out["base.feature_norm.bias"] = sd["base.feature_norm.bias"]
    srcs = ["base.mlp.fc1."] + [f"base.mlp.fc2.{i}." for i in range(cfg.layer_N)]      # fc_h is only the clone template
    for i, s in enumerate(srcs):
        out[f"base.lins.{i}.weight"] = sd[s + "0.weight"]
        out[f"base.lins.{i}.bias"] = sd[s + "0.bias"]
        out[f"base.norms.{i}.weight"] = sd[s + "2.weight"]
        out[f"base.norms.{i}.bias"] = sd[s + "2.bias"]
    if cfg.use_recurrent_policy or cfg.use_naive_recurrent_policy:
        for k, v in sd.items():
            if k.startswith("rnn."):
                out[k] = v
    if head == "actor":
        out["action_out.weight"] = sd["act.action_out.linear.weight"]
        out["action_out.bias"] = sd["act.action_out.linear.bias"]
    else:
        out["v_out.weight"] = sd["v_out.weight"]
        out["v_out.bias"] = sd["v_out.bias"]
    return out


def load_reference_state_dict(module: nn.Module, sd: Dict[str, Tensor]) -> None:
    """Load a ``GR_Actor`` / ``GR_Critic`` state dict (either EmbedConv key layout) into the dense module, strictly."""
    head = "actor" if isinstance(module, DenseGraphActor) else "critic"
    mapped = _map_reference_keys({k: torch.as_tensor(v) for k, v in sd.items()}, module.cfg, head)
    module.load_state_dict(mapped, strict=True)


def config_from_state_dict(sd: Dict[str, Any], **overrides) -> PolicyConfig:
    """Infer the shape fields of a ``PolicyConfig`` from a reference actor state dict (e.g. ``model_weights/FA/actor.pt``)."""
    e = "gnn_base.gnn.embed_layer."
    legacy = (e + "lin1.0.weight") in sd
    w1 = sd[e + ("lin1.0.weight" if legacy else "lin1.weight")]
    emb = sd[e + "entity_embed.weight"]
    key, skip = sd["gnn_base.gnn.gnn1.lin_key.weight"], sd["gnn_base.gnn.gnn1.lin_skip.weight"]
    n_embed = sum(1 for k in sd if k.startswith(e + "lin2.") and k.endswith(".0.weight")) if legacy else \
        sum(1 for k in sd if k.startswith(e + "layers.") and k.endswith(".weight") and sd[k].dim() == 2)
    n_gnn2 = len({k.split(".")[3] for k in sd if k.startswith("gnn_base.gnn.gnn2.")})
    n_mlp = sum(1 for k in sd if k.startswith("base.mlp.fc2.") and k.endswith(".0.weight"))
    hidden = sd["base.mlp.fc1.0.weight"].shape[0]
    kw = dict(
        node_feat_dim=w1.shape[1] - emb.shape[1] - 1 + 1, num_embeddings=emb.shape[0], embedding_size=emb.shape[1],
        embed_hidden_size=w1.shape[0], embed_layer_N=n_embed, gnn_layer_N=n_gnn2, hidden_size=hidden, layer_N=n_mlp,
        use_recurrent_policy=any(k.startswith("rnn.") for k in sd),
        use_feature_normalization="base.feature_norm.weight" in sd)
    concat = skip.shape[0] == key.shape[0] and key.shape[0] != skip.shape[1]
    # heads * C = key rows; C = skip rows when heads are averaged
    if concat:
        raise NotImplementedError("cannot infer heads from a concat-heads checkpoint; pass gnn_num_heads explicitly")
    kw.update(gnn_hidden_size=skip.shape[0], gnn_num_heads=key.shape[0] // skip.shape[0], gnn_concat_heads=False)
    if "act.action_out.linear.weight" in sd:
        kw.update(action_dim=sd["act.action_out.linear.weight"].shape[0],
                  obs_dim=sd["base.mlp.fc1.0.weight"].shape[1] - skip.shape[0])
    kw.update(overrides)
    return PolicyConfig(**kw)
