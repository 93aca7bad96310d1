"""Minimal stand-in for ``torch_geometric`` (TEST INFRASTRUCTURE ONLY, "parity unpinned" w.r.t. PyG).

The reference's policy (``onpolicy/algorithms/utils/gnn_new.py``, legacy twin ``gnn.py``) is built on
torch_geometric, which is not installed here and not vendored in the original project
(requirements.txt pins ``torch_geometric==2.3.1``).  To run the reference's OWN ``GNNBase`` /
``GR_Actor`` / ``GR_Critic`` code as the checker of ``fair_marl_b200.policy`` this module restates, on
edge lists with gather / index_add, the few published PyG primitives those files use:

* ``MessagePassing`` (aggr='add', flow source->target): ``x_j = x[edge_index[0]]``,
  ``x_i = x[edge_index[1]]``, ``message(...)`` per edge, sum over the incoming edges of each target.
* ``TransformerConv`` (Shi et al., "Masked Label Prediction", as implemented in PyG 2.x):
  per head ``alpha_ij = softmax_j((W_q x_i)^T (W_k x_j + W_e e_ij) / sqrt(C))``,
  ``out_i = sum_j alpha_ij (W_v x_j + W_e e_ij)``; heads concatenated or averaged; ``+ W_skip x_i``.
* segment softmax ``exp(a - max_i) / (sum_i + 1e-16)``, ``global_{mean,max,add}_pool``, ``add_self_loops``,
  ``Data``.

``install()`` registers the stand-in in ``sys.modules`` (only if the real package is absent).
There is no PyG here to pin these restatements against; DESIGN.md says so.
"""
from __future__ import annotations

import inspect
import math
import sys
import types
from typing import Optional, Tuple

import torch
from torch import Tensor, nn


def segment_softmax(src: Tensor, index: Tensor, num_segments: int) -> Tensor:
    """Softmax of ``src`` [nnz, ...] over the entries sharing ``index`` (torch_geometric.utils.softmax)."""
    shape = (num_segments,) + tuple(src.shape[1:])
    idx = index.view(-1, *([1] * (src.dim() - 1))).expand_as(src)
    mx = torch.full(shape, float("-inf"), dtype=src.dtype, device=src.device).scatter_reduce(0, idx, src, "amax")
    out = (src - mx.gather(0, idx)).exp()
    den = torch.zeros(shape, dtype=src.dtype, device=src.device).scatter_add(0, idx, out) + 1e-16
    return out / den.gather(0, idx)


class MessagePassing(nn.Module):
    """Sum aggregation over incoming edges, messages built by ``self.message`` from ``*_i`` / ``*_j`` views."""

    def __init__(self, aggr: str = "add", node_dim: int = 0, **kwargs):
        super().__init__()
        if aggr != "add":
            raise NotImplementedError("the stand-in only implements aggr='add'")
        self.aggr, self.node_dim = aggr, node_dim

    def propagate(self, edge_index: Tensor, size=None, **kwargs) -> Tensor:
        src, dst = edge_index[0], edge_index[1]
        first = next(v for v in kwargs.values() if v is not None and (isinstance(v, tuple) or v.dim() >= 1))
        num_nodes = (first[1] if isinstance(first, tuple) else first).size(0)
        feed = {}
        for name in inspect.signature(self.message).parameters:
            if name == "index":
                feed[name] = dst
            elif name == "ptr":
                feed[name] = None
            elif name == "size_i":
                feed[name] = num_nodes
            elif name.endswith("_j") or name.endswith("_i"):
                v = kwargs[name[:-2]]
                if isinstance(v, tuple):
                    v = v[0] if name.endswith("_j") else v[1]
                feed[name] = v.index_select(0, src if name.endswith("_j") else dst)
            else:
                feed[name] = kwargs.get(name)
        msg = self.message(**feed)
        out = torch.zeros((num_nodes,) + tuple(msg.shape[1:]), dtype=msg.dtype, device=msg.device)
        return out.index_add(0, dst, msg)


class TransformerConv(MessagePassing):
    def __init__(self, in_channels: int, out_channels: int, heads: int = 1, concat: bool = True, beta: bool = False,
                 dropout: float = 0.0, edge_dim: Optional[int] = None, bias: bool = True, root_weight: bool = True,
                 **kwargs):
        super().__init__(aggr="add", node_dim=0)
        if beta or dropout != 0.0 or not root_weight:
            raise NotImplementedError("the stand-in covers beta=False, dropout=0, root_weight=True (what the reference uses)")
        self.in_channels, self.out_channels, self.heads, self.concat, self.edge_dim = in_channels, out_channels, heads, concat, edge_dim
        self.lin_key = nn.Linear(in_channels, heads * out_channels)
        self.lin_query = nn.Linear(in_channels, heads * out_channels)
        self.lin_value = nn.Linear(in_channels, heads * out_channels)
        self.lin_edge = nn.Linear(edge_dim, heads * out_channels, bias=False) if edge_dim is not None else None
        self.lin_skip = nn.Linear(in_channels, heads * out_channels if concat else out_channels, bias=bias)

    def forward(self, x: Tensor, edge_index: Tensor, edge_attr: Optional[Tensor] = None) -> Tensor:
        H, C = self.heads, self.out_channels
        q = self.lin_query(x).view(-1, H, C)
        k = self.lin_key(x).view(-1, H, C)
        v = self.lin_value(x).view(-1, H, C)
        out = self.propagate(edge_index, query=q, key=k, value=v, edge_attr=edge_attr)
        out = out.view(-1, H * C) if self.concat else out.mean(dim=1)
        return out + self.lin_skip(x)

    def message(self, query_i: Tensor, key_j: Tensor, value_j: Tensor, edge_attr: Optional[Tensor], index: Tensor,
                ptr, size_i: int) -> Tensor:
        H, C = self.heads, self.out_channels
        if self.lin_edge is not None:
            e = self.lin_edge(edge_attr).view(-1, H, C)
            key_j = key_j + e
        alpha = (query_i * key_j).sum(dim=-1) / math.sqrt(C)
        alpha = segment_softmax(alpha, index, size_i)
        out = value_j + e if self.lin_edge is not None else value_j
        return out * alpha.view(-1, H, 1)


def _pool(x: Tensor, batch: Tensor, how: str) -> Tensor:
    n = int(batch.max().item()) + 1 if batch.numel() else 0
    idx = batch.view(-1, 1).expand_as(x)
    if how == "add" or how == "mean":
        out = torch.zeros((n, x.size(1)), dtype=x.dtype, device=x.device).scatter_add(0, idx, x)
        if how == "mean":
            cnt = torch.zeros(n, dtype=x.dtype, device=x.device).scatter_add(0, batch, torch.ones_like(batch, dtype=x.dtype))
            out = out / cnt.clamp(min=1).view(-1, 1)
        return out
    return torch.full((n, x.size(1)), float("-inf"), dtype=x.dtype, device=x.device).scatter_reduce(0, idx, x, "amax")


def global_mean_pool(x, batch): return _pool(x, batch, "mean")
def global_add_pool(x, batch): return _pool(x, batch, "add")
def global_max_pool(x, batch): return _pool(x, batch, "max")


def add_self_loops(edge_index: Tensor, edge_attr=None, num_nodes: Optional[int] = None) -> Tuple[Tensor, None]:
    loops = torch.arange(num_nodes, device=edge_index.device).unsqueeze(0).repeat(2, 1)
    return torch.cat([edge_index, loops], dim=1), None


class Data:
    def __init__(self, x=None, edge_index=None, edge_attr=None, batch=None, **kw):
        self.x, self.edge_index, self.edge_attr, self.batch = x, edge_index, edge_attr, batch
        self.__dict__.update(kw)


def install() -> bool:
    """Register the stand-in as ``torch_geometric`` unless the real package can be imported.  Returns True if installed."""
    try:
        import torch_geometric  # noqa: F401
        if not getattr(sys.modules["torch_geometric"], "_fairmarl_stub", False):
            return False
    except ImportError:
        pass

    def mod(name, **kw):
        m = types.ModuleType(name)
        m.__dict__.update(kw)
        m.__path__ = []
        sys.modules[name] = m
        return m

    def _unavailable(*a, **k):
        raise NotImplementedError("not part of the torch_geometric stand-in")

    from typing import Optional as Opt, Tuple as Tup, Union
    nnm = mod("torch_geometric.nn", MessagePassing=MessagePassing, TransformerConv=TransformerConv,
              global_mean_pool=global_mean_pool, global_max_pool=global_max_pool, global_add_pool=global_add_pool)
    data = mod("torch_geometric.data", Data=Data, Batch=Data, DataLoader=_unavailable)
    loader = mod("torch_geometric.loader", DataLoader=_unavailable)
    utils = mod("torch_geometric.utils", add_self_loops=add_self_loops, to_dense_batch=_unavailable, softmax=segment_softmax)
    typing_m = mod("torch_geometric.typing", OptPairTensor=Tup[Tensor, Opt[Tensor]], Adj=Tensor, OptTensor=Opt[Tensor],
                   Size=Opt[Tup[int, int]], PairTensor=Tup[Tensor, Tensor], Union=Union)
    mod("torch_geometric", nn=nnm, data=data, loader=loader, utils=utils, typing=typing_m, _fairmarl_stub=True)
    return True
