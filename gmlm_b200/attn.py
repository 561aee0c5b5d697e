"""The two aggregation variants north_star names beside the RGCN mean: GCN symmetric-degree
normalisation (SURVEY §8a row A8) and GAT edge-softmax (row A9, BASELINE.json configs[2]).
They have **no counterpart in /root/reference** (it uses only RGCNConv); semantics follow upstream
``GCNConv`` / ``GATConv`` defaults as restated in ``oracle/pyg_ref.py`` ("parity unpinned").

Both run on one dst-keyed CSR with self-loops normalised the upstream way (existing self-loops
removed, one loop per node appended).  GCN reuses the aggregation kernel ``gmlm_spmm_csr`` in weighted
mode with per-edge scalars from ``csrc/gat.cu``.  GAT is ``csrc/gat_fused.cu``: the forward is ONE pass
(online softmax, the score computed where the source row is gathered, alpha never stored), the backward
one edge pass over the same CSR plus two gathers over its transpose; long rows use the hub plan.

``GATConv(edge_dim=D)`` adds upstream's edge-feature term: a per-(edge, head) score ``alpha_edge`` (the projection
``lin_edge`` folded with ``att_edge`` into an [H, D] weight), added inside the leaky ReLU by the same kernels.
"""
from __future__ import annotations

import numbers
from collections import OrderedDict
from dataclasses import dataclass
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .graph import _LOCK, CSR, _ptr, _require_cuda, _stream, _tensor_key, build_csr, transpose_csr
from .nn import glorot_
from .ops import _dtype_code, _ld, _rowmajor, linear_nt, spmm


@dataclass
class LoopGraph:
    """dst-keyed CSR of ``edge_index`` with upstream's self-loop normalisation, plus its transpose."""
    num_nodes: int
    fwd: CSR                       # rows = dst, col = src
    bwd: CSR                       # rows = src, col = dst (row to gather the output gradient from)
    t2f: torch.Tensor              # int64 [nnz]: transposed position -> forward CSR position
    gcn_w: Optional[torch.Tensor] = None      # float32 [nnz] in forward CSR order
    gcn_w_t: Optional[torch.Tensor] = None    # same weights in transposed order
    # moving per-edge values (edge_attr) between input order and forward-CSR order without host syncs at call time
    # (csrc/gat.cu, gmlm_gat_loop_fill / _bwd):
    num_input_edges: int = 0                  # edge_index.size(1), input self-loops included
    csr_src: Optional[torch.Tensor] = None    # int32 [nnz]: input position of each CSR entry (-1 at loop entries)
    in2csr: Optional[torch.Tensor] = None     # int32 [E_in]: CSR position of each input edge (-1 for a self-loop)
    in_dst: Optional[torch.Tensor] = None     # int32 [E_in]: destination of each input edge
    loop_csr: Optional[torch.Tensor] = None   # int32 [N]: CSR position of node i's loop entry

    @staticmethod
    def build(edge_index: torch.Tensor, num_nodes: int, hub_thresh=None, quantum=None) -> "LoopGraph":
        lib = _lib.load()
        _require_cuda(edge_index, "edge_index")
        ei = edge_index.long()
        keep = ei[0] != ei[1]
        loops = torch.arange(num_nodes, dtype=torch.int64, device=ei.device)
        src = torch.cat([ei[0][keep], loops]).contiguous()         # remove_self_loops + add_self_loops
        dst = torch.cat([ei[1][keep], loops]).contiguous()
        fwd, _ = build_csr(dst, src, num_nodes, num_nodes, hub_thresh=hub_thresh, quantum=quantum)
        bwd = transpose_csr(src, dst.to(torch.int32), num_nodes, hub_thresh=hub_thresh, quantum=quantum)
        inv = torch.empty_like(fwd.perm, dtype=torch.int64)
        inv[fwd.perm.long()] = torch.arange(fwd.perm.numel(), dtype=torch.int64, device=ei.device)
        t2f = inv[bwd.perm.long()].contiguous()
        kept_pos = keep.nonzero().view(-1)                         # input positions of the kept edges
        e_kept = kept_pos.numel()
        in2csr = torch.full((ei.size(1),), -1, dtype=torch.int64, device=ei.device)
        in2csr[kept_pos] = inv[:e_kept]
        csr_src = torch.cat([kept_pos, kept_pos.new_full((num_nodes,), -1)])[fwd.perm.long()]
        g = LoopGraph(num_nodes=num_nodes, fwd=fwd, bwd=bwd, t2f=t2f, num_input_edges=int(ei.size(1)),
                      csr_src=csr_src.int(), in2csr=in2csr.int(), in_dst=ei[1].int(),
                      loop_csr=inv[e_kept:].int())
        with torch.cuda.device(ei.device):
            dis = torch.empty(num_nodes, dtype=torch.float32, device=ei.device)
            w = torch.empty(fwd.nnz, dtype=torch.float32, device=ei.device)
            _lib.check(lib.gmlm_gcn_edge_weights(_ptr(fwd.rowptr), _ptr(fwd.col), num_nodes, _ptr(dis), _ptr(w),
                                                 _stream(ei.device)), "gcn_edge_weights")
        g.gcn_w = w
        g.gcn_w_t = w[t2f].contiguous()
        return g


_LOOP_CACHE: "OrderedDict[tuple, tuple]" = OrderedDict()


def get_loop_graph(edge_index: torch.Tensor, num_nodes: int) -> LoopGraph:
    key = (_tensor_key(edge_index), int(num_nodes))
    with _LOCK:
        hit = _LOOP_CACHE.get(key)
        if hit is not None:
            _LOOP_CACHE.move_to_end(key)
            return hit[0]
        g = LoopGraph.build(edge_index, num_nodes)
        _LOOP_CACHE[key] = (g, edge_index)
        while len(_LOOP_CACHE) > 4:
            _LOOP_CACHE.popitem(last=False)
        return g


def _with_w(csr: CSR, w: torch.Tensor) -> CSR:
    """A shallow view of ``csr`` carrying different per-edge weights.  Its band plan's hub_w no longer applies, and
    without hub_w the weighted aggregation runs the CSR-order hub chunks."""
    c = CSR(**{k: getattr(csr, k) for k in csr.__dataclass_fields__})
    c.w = w
    c.hub_w = None
    return c


# ------------------------------------------------------------------------------ GCN (A8)
class _GCNAggregate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z, graph: LoopGraph):
        ctx.graph = graph
        return spmm(z, _with_w(graph.fwd, graph.gcn_w), _lib.AGG_WEIGHTED)

    @staticmethod
    def backward(ctx, g):
        graph: LoopGraph = ctx.graph
        return spmm(g.contiguous(), _with_w(graph.bwd, graph.gcn_w_t), _lib.AGG_WEIGHTED), None


class GCNConv(nn.Module):
    """Upstream ``GCNConv`` defaults: ``out = D^-1/2 (A + I) D^-1/2 (x W) + b`` (row A8)."""

    def __init__(self, in_channels: int, out_channels: int, bias: bool = True):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin = nn.Linear(in_channels, out_channels, bias=False)
        if bias:
            self.bias = nn.Parameter(torch.zeros(out_channels))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        glorot_(self.lin.weight)
        if self.bias is not None:
            nn.init.zeros_(self.bias)

    def forward(self, x: torch.Tensor, edge_index) -> torch.Tensor:
        graph = edge_index if isinstance(edge_index, LoopGraph) else get_loop_graph(edge_index, x.size(0))
        out = _GCNAggregate.apply(self.lin(x), graph)
        return out + self.bias if self.bias is not None else out


# ------------------------------------------------------------------------------ GAT (A9)
def _hub_args(csr: CSR):
    return (csr.hub_thresh, csr.n_hub, csr.n_chunks, _ptr(csr.hub_row), _ptr(csr.hub_chunk_ptr), _ptr(csr.chunk_beg),
            _ptr(csr.chunk_end))


def _check_a_edge(a_edge, graph: LoopGraph, heads: int):
    if a_edge is not None and (a_edge.shape != (graph.fwd.nnz, heads) or a_edge.dtype != torch.float32
                               or not a_edge.is_contiguous()):
        raise _lib.GmlmError(f"gat: a_edge must be a contiguous float32 [nnz = {graph.fwd.nnz}, heads = {heads}] "
                             f"tensor in forward-CSR order, got {a_edge.dtype} {tuple(a_edge.shape)}")


def _gat_forward(z, a_src32, a_dst32, graph: LoopGraph, slope: float, p_drop: float, seed: int,
                 a_edge: Optional[torch.Tensor] = None):
    """The fused forward (csrc/gat_fused.cu) on row-major ``z`` (any leading dimension): ``(out, m, l)``.
    ``a_edge``: optional fp32 [nnz, H] score term in forward-CSR order (None: the kernels without it)."""
    lib = _lib.load()
    n, heads = a_dst32.shape
    head_dim = z.size(1) // heads
    dev = z.device
    fwd = graph.fwd
    _check_a_edge(a_edge, graph, heads)
    with torch.cuda.device(dev):
        out = torch.empty((n, heads * head_dim), dtype=z.dtype, device=dev)
        m = torch.empty((n, heads), dtype=torch.float32, device=dev)
        l = torch.empty((n, heads), dtype=torch.float32, device=dev)
        ws_bytes = lib.gmlm_gat_workspace_bytes(fwd.n_chunks, heads, head_dim) if fwd.n_hub else 0
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
        _lib.check(lib.gmlm_gat_fused_fwd_eattr(_ptr(fwd.rowptr), _ptr(fwd.col), n, _ptr(z), _dtype_code(z, "gat"),
                                                _ld(z), _ptr(a_src32), _ptr(a_dst32), _ptr(a_edge), heads, head_dim,
                                                float(slope), float(p_drop), int(seed), *_hub_args(fwd), _ptr(ws),
                                                ws_bytes, _ptr(out), heads * head_dim, _ptr(m), _ptr(l), _stream(dev)),
                   "gat_fused_fwd")
    return out, m, l


def _gat_backward(g, z, a_src, a_dst, m, l, out, graph: LoopGraph, slope: float, p_drop: float, seed: int,
                  dz_out: Optional[torch.Tensor] = None, a_edge: Optional[torch.Tensor] = None):
    """``(dz, da_src, da_dst, d_score)`` of the fused forward; ``da_*`` and ``d_score`` fp32, ``d_score`` [nnz, H] in
    forward-CSR order (the gradient of the raw score, and so of ``a_edge``).  ``dz_out``: a row-major [N, H*C] view
    (any leading dimension, e.g. the first columns of a wider gradient) that receives dz instead of a new tensor."""
    lib = _lib.load()
    fwd = graph.fwd
    n, heads = a_dst.shape
    head_dim = z.size(1) // heads
    dev = z.device
    # t[i,h] = <g[i,h,:], out[i,h,:]> = sum_e alpha_e keep_e d_alpha_e (no pass over the edges needed)
    t = (g.view(n, heads, head_dim).float() * out.view(n, heads, head_dim).float()).sum(-1).contiguous()
    with torch.cuda.device(dev):
        alpha_eff = torch.empty((fwd.nnz, heads), dtype=torch.float32, device=dev)
        d_score = torch.empty((fwd.nnz, heads), dtype=torch.float32, device=dev)
        da_dst = torch.empty((n, heads), dtype=torch.float32, device=dev)
        ws_bytes = lib.gmlm_gat_workspace_bytes(fwd.n_chunks, heads, head_dim) if fwd.n_hub else 0
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
        _lib.check(lib.gmlm_gat_bwd_edges_eattr(_ptr(fwd.rowptr), _ptr(fwd.col), n, _ptr(z), _dtype_code(z, "gat"),
                                                _ld(z), _ptr(g), _ld(g), _ptr(a_src), _ptr(a_dst), _ptr(a_edge), _ptr(m),
                                                _ptr(l), _ptr(t), heads, head_dim, slope, p_drop, seed,
                                                *_hub_args(fwd), _ptr(ws), ws_bytes, _ptr(alpha_eff), _ptr(d_score),
                                                _ptr(da_dst), _stream(dev)),
                   "gat_bwd_edges")
        da_src = torch.empty((a_src.size(0), heads), dtype=torch.float32, device=dev)
        _lib.check(lib.gmlm_segment_sum_f32(_ptr(d_score), _ptr(graph.t2f), _ptr(graph.bwd.rowptr), a_src.size(0),
                                            heads, _ptr(da_src), _stream(dev)), "segment_sum")
    dz = spmm(g, _with_w(graph.bwd, alpha_eff[graph.t2f].contiguous()), _lib.AGG_WEIGHTED, out=dz_out)
    return dz, da_src, da_dst, d_score


class _GATAggregate(torch.autograd.Function):
    """Fused edge-softmax aggregation (csrc/gat_fused.cu): one pass, online softmax, alpha never stored."""

    @staticmethod
    def forward(ctx, z, a_src, a_dst, graph: LoopGraph, slope: float, p_drop: float, seed: int,
                a_edge: Optional[torch.Tensor] = None):
        z = _rowmajor(z)
        a_src32, a_dst32 = a_src.detach().float().contiguous(), a_dst.detach().float().contiguous()
        a_edge32 = a_edge.detach().float().contiguous() if a_edge is not None else None
        out, m, l = _gat_forward(z, a_src32, a_dst32, graph, slope, p_drop, seed, a_edge32)
        ctx.graph, ctx.slope, ctx.p_drop, ctx.seed = graph, float(slope), float(p_drop), int(seed)
        ctx.save_for_backward(z, a_src32, a_dst32, m, l, out, a_edge32)
        ctx.in_dtypes = (a_src.dtype, a_dst.dtype, a_edge.dtype if a_edge is not None else None)
        return out

    @staticmethod
    def backward(ctx, g):
        z, a_src, a_dst, m, l, out, a_edge = ctx.saved_tensors
        g = _rowmajor(g)
        if g.dtype != z.dtype:
            g = g.to(z.dtype)
        dz, da_src, da_dst, d_score = _gat_backward(g, z, a_src, a_dst, m, l, out, ctx.graph, ctx.slope, ctx.p_drop,
                                                    ctx.seed, a_edge=a_edge)
        d_edge = d_score.to(ctx.in_dtypes[2]) if a_edge is not None and ctx.needs_input_grad[7] else None
        return dz, da_src.to(ctx.in_dtypes[0]), da_dst.to(ctx.in_dtypes[1]), None, None, None, None, d_edge


class _GATAggregateScored(torch.autograd.Function):
    """The aggregation fed by ONE projection ``y = x @ [W ; w_src ; w_dst]^T`` (``gat_score_weight``):
    ``z = y[:, :H*C]`` is read in place (leading dimension = y's), ``a_src`` / ``a_dst`` are y's next 2H columns.
    The backward writes dz, da_src and da_dst straight into the columns of one gradient buffer shaped like y, so
    nothing assembles the GEMM's output gradient in a separate pass."""

    @staticmethod
    def forward(ctx, y, heads: int, graph: LoopGraph, slope: float, p_drop: float, seed: int,
                a_edge: Optional[torch.Tensor] = None):
        y = _rowmajor(y)
        hc = y.size(1) - 2 * heads
        z = y[:, :hc]
        a_src32 = y[:, hc:hc + heads].contiguous()
        a_dst32 = y[:, hc + heads:].contiguous()
        a_edge32 = a_edge.detach().float().contiguous() if a_edge is not None else None
        out, m, l = _gat_forward(z, a_src32, a_dst32, graph, slope, p_drop, seed, a_edge32)
        ctx.graph, ctx.slope, ctx.p_drop, ctx.seed, ctx.heads = graph, float(slope), float(p_drop), int(seed), heads
        ctx.save_for_backward(y, a_src32, a_dst32, m, l, out, a_edge32)
        return out

    @staticmethod
    def backward(ctx, g):
        y, a_src, a_dst, m, l, out, a_edge = ctx.saved_tensors
        heads = ctx.heads
        hc = y.size(1) - 2 * heads
        g = _rowmajor(g)
        if g.dtype != y.dtype:
            g = g.to(y.dtype)
        n, width = y.shape
        per = 4                                   # fp32: 16-byte row pitch, as the GEMM lays out y
        dy = torch.empty((n, (width + per - 1) // per * per), dtype=y.dtype, device=y.device)[:, :width]
        _, da_src, da_dst, d_score = _gat_backward(g, y[:, :hc], a_src, a_dst, m, l, out, ctx.graph, ctx.slope,
                                                   ctx.p_drop, ctx.seed, dz_out=dy[:, :hc], a_edge=a_edge)
        dy[:, hc:hc + heads].copy_(da_src)
        dy[:, hc + heads:].copy_(da_dst)
        d_edge = d_score if a_edge is not None and ctx.needs_input_grad[6] else None
        return dy, None, None, None, None, None, d_edge


def gat_aggregate(z, a_src, a_dst, graph: LoopGraph, negative_slope: float = 0.2, dropout: float = 0.0,
                  seed: int = 0, a_edge: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``out[i,h,:] = sum_j softmax_j(leaky_relu(a_src[j,h] + a_dst[i,h])) * z[j,h,:]`` over the in-edges, with
    optional attention dropout (keep mask = counter-based hash of (seed, edge, head): see ``gat_dropout_mask``).
    ``a_edge``: optional fp32 [nnz, H] term added to the score of every edge, in forward-CSR order with the self-loop
    entries (``graph.fwd``); its gradient is the score gradient."""
    _require_cuda(z, "z")
    return _GATAggregate.apply(z, a_src, a_dst, graph, negative_slope, dropout, seed, a_edge)


class _EdgeScoresCSR(torch.autograd.Function):
    """Per-edge scores in input order ``alpha [E_in, H]`` -> ``a_edge [nnz, H]`` in forward-CSR order: the rows of
    the kept (non-loop) edges, and at each node's loop entry the mean over its kept in-edges (upstream
    ``add_self_loops(fill_value="mean")``; 0 for a node without in-edges).  Input self-loops drop out with their rows.
    One kernel each way (csrc/gat.cu): a warp per CSR row forward, a thread per (input edge, head) backward.  No
    atomics, no host syncs."""

    @staticmethod
    def forward(ctx, alpha, graph: LoopGraph):
        lib = _lib.load()
        heads = alpha.size(1)
        dev = alpha.device
        alpha = alpha.detach().float().contiguous()
        fwd = graph.fwd
        with torch.cuda.device(dev):
            a = torch.empty((fwd.nnz, heads), dtype=torch.float32, device=dev)
            _lib.check(lib.gmlm_gat_loop_fill(_ptr(alpha), _ptr(graph.csr_src), _ptr(graph.loop_csr),
                                              _ptr(fwd.rowptr), graph.num_nodes, heads, _ptr(a), _stream(dev)),
                       "gat_loop_fill")
        ctx.graph = graph
        return a

    @staticmethod
    def backward(ctx, g):
        lib = _lib.load()
        graph: LoopGraph = ctx.graph
        g = g.float().contiguous()
        dev = g.device
        with torch.cuda.device(dev):
            d = torch.empty((graph.num_input_edges, g.size(1)), dtype=torch.float32, device=dev)
            _lib.check(lib.gmlm_gat_loop_fill_bwd(_ptr(g), _ptr(graph.in2csr), _ptr(graph.in_dst),
                                                  _ptr(graph.loop_csr), _ptr(graph.fwd.rowptr),
                                                  graph.num_input_edges, g.size(1), _ptr(d), _stream(dev)),
                       "gat_loop_fill_bwd")
        return d, None


def gat_edge_scores(alpha: torch.Tensor, graph: LoopGraph) -> torch.Tensor:
    """fp32 ``[E_in, H]`` per-edge scores of ``edge_index``'s edges (input order) -> the ``a_edge [nnz, H]`` of
    ``gat_aggregate``: input self-loops dropped, one loop per node filled with the mean of its in-edges' scores."""
    _require_cuda(alpha, "alpha")
    if alpha.dim() != 2 or alpha.size(0) != graph.num_input_edges:
        raise ValueError(f"gat_edge_scores: expected [{graph.num_input_edges}, heads] scores (one row per input "
                         f"edge), got {tuple(alpha.shape)}")
    return _EdgeScoresCSR.apply(alpha, graph)


def gat_score_weight(weight: torch.Tensor, att_src: torch.Tensor, att_dst: torch.Tensor) -> torch.Tensor:
    """``[W ; w_src ; w_dst]`` [H*C + 2H, K]: the projection weight with the attention vectors folded in, so that
    ``x @ W_ext^T = [z | a_src | a_dst]`` with ``a_src[i,h] = sum_c z[i,h,c] att_src[h,c]`` (and ``a_dst`` likewise),
    because ``a_src[i,h] = x_i . (sum_c att_src[h,c] W[h*C+c, :])``.  Differentiable in all three parameters."""
    heads, c = att_src.shape[-2], att_src.shape[-1]
    wv = weight.view(heads, c, weight.size(1))
    w_src = torch.einsum("hc,hck->hk", att_src.reshape(heads, c), wv)
    w_dst = torch.einsum("hc,hck->hk", att_dst.reshape(heads, c), wv)
    return torch.cat([weight, w_src, w_dst], dim=0)


def gat_edge_weight(lin_edge_weight: torch.Tensor, att_edge: torch.Tensor) -> torch.Tensor:
    """``w_edge [H, D]``, ``w_edge[h,d] = sum_c att_edge[h,c] lin_edge.weight[h*C+c, d]``: upstream's
    ``alpha_edge = (lin_edge(edge_attr).view(E, H, C) * att_edge).sum(-1)`` is ``edge_attr @ w_edge.T``, without the
    [E, H*C] projection.  Differentiable in both parameters."""
    heads, c = att_edge.shape[-2], att_edge.shape[-1]
    wv = lin_edge_weight.view(heads, c, lin_edge_weight.size(1))
    return torch.einsum("hc,hcd->hd", att_edge.reshape(heads, c), wv)


def gat_dropout_mask(seed: int, num_edges: int, heads: int, p_drop: float, device) -> torch.Tensor:
    """bool [num_edges, heads] keep mask of the fused kernels, edges in forward-CSR order (tests / inspection)."""
    lib = _lib.load()
    dev = torch.device(device)
    with torch.cuda.device(dev):
        keep = torch.empty(num_edges * heads, dtype=torch.uint8, device=dev)
        _lib.check(lib.gmlm_gat_dropout_mask(int(seed), keep.numel(), float(p_drop), _ptr(keep), _stream(dev)),
                   "gat_dropout_mask")
    return keep.view(num_edges, heads).bool()


class GATConv(nn.Module):
    """Upstream ``GATConv`` defaults (self-loops, LeakyReLU 0.2, concat heads, bias, attention dropout in training
    mode).  Row A9 / BASELINE configs[2].  The edge-softmax and the aggregation are ONE kernel pass.

    ``edge_dim = D`` adds upstream's edge features: ``lin_edge`` (Linear(D, H*C), no bias) and ``att_edge [1, H, C]``,
    and ``forward(x, edge_index, edge_attr)`` adds ``alpha_edge[e,h] = sum_c lin_edge(edge_attr)[e,h,c] att_edge[h,c]``
    to the score inside the leaky ReLU.  Input self-loops are dropped with their attributes; each node's loop gets
    the mean of its in-edges' attributes (``fill_value="mean"``, the only fill supported).  Without ``edge_dim`` an
    ``edge_attr`` is ignored, as upstream does."""

    def __init__(self, in_channels: int, out_channels: int, heads: int = 1, concat: bool = True,
                 negative_slope: float = 0.2, dropout: float = 0.0, bias: bool = True,
                 edge_dim: Optional[int] = None, fill_value="mean"):
        super().__init__()
        if not 0.0 <= dropout < 1.0:
            raise ValueError("gmlm_b200.GATConv: dropout must be in [0, 1)")
        if not (isinstance(fill_value, str) and fill_value == "mean"):
            raise NotImplementedError(f"gmlm_b200.GATConv: fill_value={fill_value!r}; only 'mean' is supported")
        self.in_channels, self.out_channels, self.heads, self.concat = in_channels, out_channels, heads, concat
        self.negative_slope = negative_slope
        self.dropout = dropout
        self.edge_dim, self.fill_value = edge_dim, fill_value
        self.lin = nn.Linear(in_channels, heads * out_channels, bias=False)
        self.att_src = nn.Parameter(torch.empty(1, heads, out_channels))
        self.att_dst = nn.Parameter(torch.empty(1, heads, out_channels))
        if edge_dim is not None:
            self.lin_edge = nn.Linear(edge_dim, heads * out_channels, bias=False)
            self.att_edge = nn.Parameter(torch.empty(1, heads, out_channels))
        else:
            self.lin_edge = None
            self.register_parameter("att_edge", None)
        if bias:
            self.bias = nn.Parameter(torch.zeros(heads * out_channels if concat else out_channels))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        glorot_(self.lin.weight)
        glorot_(self.att_src)
        glorot_(self.att_dst)
        if self.lin_edge is not None:
            glorot_(self.lin_edge.weight)
            glorot_(self.att_edge)
        if self.bias is not None:
            nn.init.zeros_(self.bias)

    def _edge_scores(self, edge_attr: torch.Tensor, graph: LoopGraph) -> torch.Tensor:
        """``a_edge [nnz, H]`` fp32 in forward-CSR order from ``edge_attr [E, D]`` (or [E] for D = 1), outside
        autocast: the folded projection ``edge_attr @ w_edge.T`` per input edge, then the loop fill."""
        ea = edge_attr.view(-1, 1) if edge_attr.dim() == 1 else edge_attr
        if ea.dim() != 2 or ea.size(0) != graph.num_input_edges or ea.size(1) != self.edge_dim:
            raise ValueError(f"gmlm_b200.GATConv: edge_attr must be [num_edges = {graph.num_input_edges}, "
                             f"edge_dim = {self.edge_dim}], got {tuple(edge_attr.shape)}")
        with torch.amp.autocast("cuda", enabled=False):
            w_edge = gat_edge_weight(self.lin_edge.weight, self.att_edge).float()
            return gat_edge_scores(F.linear(ea.float(), w_edge), graph)

    def forward(self, x: torch.Tensor, edge_index, edge_attr: Optional[torch.Tensor] = None,
                dropout_seed: Optional[int] = None) -> torch.Tensor:
        if edge_attr is not None and not isinstance(edge_attr, torch.Tensor):
            raise TypeError(f"gmlm_b200.GATConv.forward: edge_attr must be a tensor or None, got "
                            f"{type(edge_attr).__name__}; pass a dropout seed by keyword (dropout_seed=...)")
        if dropout_seed is not None and (isinstance(dropout_seed, (bool, torch.Tensor))
                                         or not isinstance(dropout_seed, numbers.Integral)):
            raise TypeError(f"gmlm_b200.GATConv.forward: dropout_seed must be an int or None, got "
                            f"{type(dropout_seed).__name__}; edge features go in edge_attr, the third argument")
        n, h, c = x.size(0), self.heads, self.out_channels
        graph = edge_index if isinstance(edge_index, LoopGraph) else get_loop_graph(edge_index, n)
        a_edge = self._edge_scores(edge_attr, graph) if self.lin_edge is not None and edge_attr is not None else None
        p = self.dropout if self.training else 0.0
        seed = 0
        if p > 0.0:                      # one draw from torch's CPU generator per call (reproducible under manual_seed)
            seed = int(dropout_seed) if dropout_seed is not None else int(torch.randint(0, 2 ** 62, (1,)).item())
        op = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else None
        if op in (torch.float16, torch.bfloat16) and x.is_cuda:
            # autocast (the reference's training loops, main.py:446,543): ONE tcgen05 GEMM with 16-bit operands and
            # fp32 results writes [z | a_src | a_dst]; the aggregation runs on fp32 z
            with torch.amp.autocast("cuda", enabled=False):
                w_ext = gat_score_weight(self.lin.weight, self.att_src, self.att_dst)
                y = linear_nt(x, w_ext, out_dtype=torch.float32, op_dtype=op)
                out = _GATAggregateScored.apply(y, h, graph, self.negative_slope, p, seed, a_edge)
        else:
            z = self.lin(x)
            zv = z.view(n, h, c)
            a_src = (zv * self.att_src).sum(-1)
            a_dst = (zv * self.att_dst).sum(-1)
            out = gat_aggregate(z, a_src, a_dst, graph, self.negative_slope, p, seed, a_edge=a_edge)
        if not self.concat:
            out = out.view(n, h, c).mean(dim=1)
        return out + self.bias if self.bias is not None else out
