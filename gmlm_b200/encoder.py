"""The GNN encoder of the reference (``GraphTextLM.get_graph_embeddings``,
``/root/reference/main.py:250-320``) on the CUDA path, with the reference's submodule names
(``rgcn1..4``, ``gnorm1..4``, ``dropout1..4``, ``residual_proj1..3``, ``multi_scale_fusion``,
``gnn_mask_token_embed``) so its state dict can be loaded into / out of ``GraphTextLM``.

What changes relative to the reference body (results stay within the parity tolerances):
  * edge typing (main.py:253-267) is one kernel and is cached per ``edge_index`` — the
    reference recomputes it with a per-edge Python loop on every call;
  * the typed CSR is built once per graph instead of five mask compactions per layer call;
  * GraphNorm + GELU run as one fused pass (two passes in backward);
  * the dead ``x4 + residual_proj3(x2)`` (main.py:317-318) is not computed — its result is
    discarded by the reference, so ``residual_proj3`` gets no gradient there either;
  * activation checkpointing (main.py:278) stays available (``use_checkpoint=True``) and is
    re-entrant-safe: the ops use no RNG and the graph cache is read-only.

``conv="gat"`` builds the same body on GAT edge-softmax layers (BASELINE configs[2]): ``gat1..gat4`` =
``GATConv(dims[k], dims[k+1] // heads, heads)`` with concatenated heads and attention dropout 0 in place of
``rgcn1..rgcn4``; every other submodule keeps its name and code.  The four layers share one self-looped CSR
(``get_loop_graph``); no edge types are computed.  fp32 activations only (eval mode, or autocast with fp32 results).
``gat_edge_types=True`` gives the GAT layers the RGCN encoder's relations as edge features: ``gatK =
GATConv(..., edge_dim=num_relations)``, fed the one-hot of the degree-bucket edge types (cached per graph), so the
attention score of every edge carries a learned per-relation, per-head term.
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.utils.checkpoint import checkpoint

from .graph import _LOCK, _tensor_key, get_rel_graph
from .attn import GATConv, get_loop_graph
from .nn import GraphNorm, RGCNConv
from .ops import edge_type_from_degree, layer_norm, layer_norm_ok, linear_nt, soft_masking_gnn_input


class MultiScaleFusion(nn.Module):
    """``MultiScaleFusion`` of main.py:167-180 (dense; stock PyTorch, ends the encoder region)."""

    def __init__(self, hidden_dims, output_dim):
        super().__init__()
        self.scale_weights = nn.Parameter(torch.ones(len(hidden_dims)) / len(hidden_dims))
        self.projections = nn.ModuleList([nn.Linear(d, output_dim) for d in hidden_dims])
        self.layer_norm = nn.LayerNorm(output_dim)

    def forward(self, embeddings_list):
        # sum_l w_l (x_l W_l^T + b_l)  ==  [x_1 | .. | x_4] @ [w_1 W_1 | .. | w_4 W_4]^T + sum_l w_l b_l :
        # one GEMM over the concatenated layer outputs instead of four projections, four broadcast
        # multiplies by a 0-dim weight and three adds over [N, out_dim] (26 % of the encoder step on
        # the 2M-node graph went into those elementwise passes)
        w = F.softmax(self.scale_weights, dim=0)
        dt = self.projections[0].weight.dtype
        autocast = torch.is_autocast_enabled("cuda")
        with torch.amp.autocast("cuda", enabled=False):
            weight = torch.cat([w[i] * p.weight for i, p in enumerate(self.projections)], dim=1)
            bias = sum(w[i] * p.bias for i, p in enumerate(self.projections))
        op = _dense_op_dtype(embeddings_list[0])
        if op is not None and len(embeddings_list) <= 4 and embeddings_list[0].is_cuda:
            # the tcgen05 GEMM reads the layer outputs through one tensor map each: no concatenation (csrc/gemm_tcgen05.cu)
            with torch.amp.autocast("cuda", enabled=False):
                fused = linear_nt(list(embeddings_list), weight, bias, op_dtype=op,
                                  out_dtype=torch.float32 if autocast else embeddings_list[0].dtype)
        else:
            xs = torch.cat([e if autocast else e.to(dt) for e in embeddings_list], dim=1)
            fused = F.linear(xs, weight, bias)
        ln = self.layer_norm
        if autocast:                      # torch.autocast runs layer_norm in fp32
            fused = fused.float()
        if ln.elementwise_affine and ln.bias is not None and layer_norm_ok(fused):
            return layer_norm(fused, ln.weight, ln.bias, ln.eps)     # row-wise kernel (csrc/layernorm.cu)
        return ln(fused)                  # widths the kernel does not take: stock, as in the reference


def _dense_op_dtype(x: torch.Tensor) -> Optional[torch.dtype]:
    """Operand type of a dense projection on the tcgen05 GEMM: the autocast type under torch.amp.autocast, bf16 in
    the bf16 pipeline; None = fp32 activations outside autocast (stock cuBLAS path)."""
    if torch.is_autocast_enabled("cuda"):
        dt = torch.get_autocast_dtype("cuda")
        return dt if dt in (torch.float16, torch.bfloat16) else None
    return torch.bfloat16 if x.dtype == torch.bfloat16 else None


_ET_CACHE: "OrderedDict[tuple, tuple]" = OrderedDict()
_ONEHOT_CACHE: "OrderedDict[tuple, tuple]" = OrderedDict()


def cached_edge_type(edge_index: torch.Tensor, num_nodes: int) -> torch.Tensor:
    """Degree-bucket relation ids for ``edge_index`` (main.py:253-267), computed once per graph.  Keyed on the
    identity of ``edge_index`` (the reference passes the same ``data.edge_index`` every call); the SAME tensor is
    returned on a hit, so the graph cache behind it hits on identity as well."""
    key = (_tensor_key(edge_index), int(num_nodes))
    with _LOCK:                                    # autograd threads recompute checkpointed layers
        hit = _ET_CACHE.get(key)
        if hit is not None:
            _ET_CACHE.move_to_end(key)
            return hit[0]
        et = edge_type_from_degree(edge_index, num_nodes)
        _ET_CACHE[key] = (et, edge_index)          # keep the key tensor alive (see graph.py cache note)
        while len(_ET_CACHE) > 4:
            _ET_CACHE.popitem(last=False)
        return et


def cached_edge_type_onehot(edge_type: torch.Tensor, num_relations: int) -> torch.Tensor:
    """float32 ``[E, num_relations]`` one-hot of ``edge_type`` (the ``edge_attr`` of the typed GAT encoder), built
    once per edge-type tensor and keyed on its identity like ``cached_edge_type``, so no encoder call allocates it."""
    key = (_tensor_key(edge_type), int(num_relations))
    with _LOCK:
        hit = _ONEHOT_CACHE.get(key)
        if hit is not None:
            _ONEHOT_CACHE.move_to_end(key)
            return hit[0]
        oh = F.one_hot(edge_type.long(), num_relations).float()
        _ONEHOT_CACHE[key] = (oh, edge_type)
        while len(_ONEHOT_CACHE) > 4:
            _ONEHOT_CACHE.popitem(last=False)
        return oh


class GraphEncoder(nn.Module):
    def __init__(self, gnn_in_channels: int, hidden_channels: int, out_dim: int, num_relations: int = 5,
                 num_bases: int = 30, dropout_rate: float = 0.3, use_checkpoint: bool = False,
                 act_dtype: Optional[torch.dtype] = None, conv: str = "rgcn", heads: int = 8,
                 gat_edge_types: bool = False):
        super().__init__()
        h = hidden_channels
        dims = [gnn_in_channels, h, 2 * h, 4 * h, 8 * h]
        if conv not in ("rgcn", "gat"):
            raise ValueError(f"GraphEncoder: conv must be 'rgcn' or 'gat', got {conv!r}")
        if gat_edge_types and conv != "gat":
            raise ValueError("GraphEncoder: gat_edge_types applies to conv='gat' only")
        if conv == "gat":
            if heads < 1 or any(d % heads for d in dims[1:]):
                raise ValueError(f"GraphEncoder: heads = {heads} must divide every GAT layer width {dims[1:]}")
            if act_dtype == torch.bfloat16:
                raise NotImplementedError("GraphEncoder: the GAT encoder runs fp32 activations (eval or autocast), "
                                          "not the bf16 pipeline")
        self.dims = dims
        self.conv = conv
        self.gat_edge_types = bool(gat_edge_types)
        self.gnn_mask_token_embed = nn.Parameter(torch.zeros(1, gnn_in_channels))   # main.py:185-186
        nn.init.xavier_uniform_(self.gnn_mask_token_embed)
        for k in range(4):                                                          # main.py:189-203
            if conv == "gat":
                setattr(self, f"gat{k+1}", GATConv(dims[k], dims[k + 1] // heads, heads=heads,
                                                   edge_dim=num_relations if gat_edge_types else None))
            else:
                setattr(self, f"rgcn{k+1}", RGCNConv(dims[k], dims[k + 1], num_relations=num_relations,
                                                     num_bases=num_bases, out_dtype=act_dtype))
            setattr(self, f"gnorm{k+1}", GraphNorm(dims[k + 1]))
            setattr(self, f"dropout{k+1}", nn.Dropout(dropout_rate))
        self.residual_proj1 = nn.Linear(gnn_in_channels, h)                         # main.py:205-207
        self.residual_proj2 = nn.Linear(h, 2 * h)
        self.residual_proj3 = nn.Linear(2 * h, 8 * h)
        self.multi_scale_fusion = MultiScaleFusion(dims[1:], out_dim)
        self.num_relations = num_relations
        self.use_checkpoint = use_checkpoint

    def _block(self, k: int):
        conv, norm, drop = getattr(self, f"{self.conv}{k}"), getattr(self, f"gnorm{k}"), getattr(self, f"dropout{k}")

        def run(x, graph, *edge_attr):
            y = conv(x, graph, *edge_attr)
            if y.size(0) > 1:                       # main.py:273
                y = norm(y, fuse_gelu=True)         # GraphNorm + exact-erf GELU in one pass
            else:
                y = F.gelu(y)
            return drop(y)
        return run

    def _run(self, k, x, graph, *edge_attr):
        if self.use_checkpoint and torch.is_grad_enabled():
            return checkpoint(self._block(k), x, graph, *edge_attr, use_reentrant=False)
        return self._block(k)(x, graph, *edge_attr)

    def _residual(self, lin: nn.Linear, x: torch.Tensor, acc: torch.Tensor) -> torch.Tensor:
        """``acc + lin(x)`` (main.py:281-282, 294-295).  On the tcgen05 GEMM the add happens in the epilogue: the
        projection reads ``acc`` tile by tile and writes the sum, no separate elementwise pass."""
        op = _dense_op_dtype(x)
        if op is not None and x.is_cuda and acc.dtype in (torch.float32, torch.bfloat16):
            with torch.amp.autocast("cuda", enabled=False):
                return linear_nt(x, lin.weight, lin.bias, out_dtype=acc.dtype, op_dtype=op, addend=acc)
        if x.dtype == lin.weight.dtype:
            return acc + lin(x).to(acc.dtype)
        return acc + F.linear(x, lin.weight.to(x.dtype), lin.bias.to(x.dtype)).to(acc.dtype)

    def get_graph_embeddings(self, x_feat: torch.Tensor, edge_index: torch.Tensor,
                             edge_type: Optional[torch.Tensor] = None, return_layers: bool = False):
        n = x_feat.size(0)
        ea = ()                                       # the GAT layers' edge_attr, when they take edge types
        if self.conv == "gat":
            graph = get_loop_graph(edge_index, n)     # edge_type is not used by GAT layers without gat_edge_types
            if self.gat_edge_types:
                if edge_type is None:
                    edge_type = cached_edge_type(edge_index, n)
                ea = (cached_edge_type_onehot(edge_type, self.num_relations),)
        else:
            if edge_type is None:
                edge_type = cached_edge_type(edge_index, n)
            graph = get_rel_graph(edge_index, edge_type, n, self.num_relations)
        outs = []
        x1 = self._run(1, x_feat, graph, *ea)
        outs.append(x1)                              # pre-residual outputs feed the fusion (main.py:279)
        x1 = self._residual(self.residual_proj1, x_feat, x1)
        x2 = self._run(2, x1, graph, *ea)
        outs.append(x2)
        x2 = self._residual(self.residual_proj2, x1, x2)
        x3 = self._run(3, x2, graph, *ea)
        outs.append(x3)
        x4 = self._run(4, x3, graph, *ea)
        outs.append(x4)
        fused = self.multi_scale_fusion(outs)
        return (fused, outs) if return_layers else fused

    def forward(self, x_feat, edge_index, edge_type=None, gnn_perturb_mask: Optional[torch.Tensor] = None,
                beta: float = 0.7):
        """Optionally applies the soft node masking of main.py:92-99 first (callers main.py:443,541)."""
        if gnn_perturb_mask is not None:
            x_feat = soft_masking_gnn_input(x_feat, gnn_perturb_mask, self.gnn_mask_token_embed, beta)
        return self.get_graph_embeddings(x_feat, edge_index, edge_type)
