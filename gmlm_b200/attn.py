"""The two aggregation variants north_star names beside the RGCN mean: GCN symmetric-degree
normalisation (SURVEY §8a row A8) and GAT edge-softmax (row A9, BASELINE.json configs[2]).
They have **no counterpart in /root/reference** (it uses only RGCNConv); semantics follow upstream
``GCNConv`` / ``GATConv`` defaults as restated in ``oracle/pyg_ref.py`` ("parity unpinned").

Both run on one dst-keyed CSR with self-loops normalised the upstream way (existing self-loops
removed, one loop per node appended).  GCN reuses the aggregation kernel ``gmlm_spmm_csr`` in weighted
mode with per-edge scalars from ``csrc/gat.cu``.  GAT is ``csrc/gat_fused.cu``: the forward is ONE pass
(online softmax, the score computed where the source row is gathered, alpha never stored), the backward
one edge pass over the same CSR plus two gathers over its transpose; long rows use the hub plan.
"""
from __future__ import annotations

from collections import OrderedDict
from dataclasses import dataclass
from typing import Optional

import torch
import torch.nn as nn

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
        g = LoopGraph(num_nodes=num_nodes, fwd=fwd, bwd=bwd, t2f=t2f)
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
    """A shallow view of ``csr`` carrying different per-edge weights (its band plan's hub_w no longer applies)."""
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


def _gat_forward(z, a_src32, a_dst32, graph: LoopGraph, slope: float, p_drop: float, seed: int):
    """The fused forward (csrc/gat_fused.cu) on row-major ``z`` (any leading dimension): ``(out, m, l)``."""
    lib = _lib.load()
    n, heads = a_dst32.shape
    head_dim = z.size(1) // heads
    dev = z.device
    fwd = graph.fwd
    with torch.cuda.device(dev):
        out = torch.empty((n, heads * head_dim), dtype=z.dtype, device=dev)
        m = torch.empty((n, heads), dtype=torch.float32, device=dev)
        l = torch.empty((n, heads), dtype=torch.float32, device=dev)
        ws_bytes = lib.gmlm_gat_workspace_bytes(fwd.n_chunks, heads, head_dim) if fwd.n_hub else 0
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
        _lib.check(lib.gmlm_gat_fused_fwd(_ptr(fwd.rowptr), _ptr(fwd.col), n, _ptr(z), _dtype_code(z, "gat"), _ld(z),
                                          _ptr(a_src32), _ptr(a_dst32), heads, head_dim, float(slope), float(p_drop),
                                          int(seed), *_hub_args(fwd), _ptr(ws), ws_bytes, _ptr(out),
                                          heads * head_dim, _ptr(m), _ptr(l), _stream(dev)), "gat_fused_fwd")
    return out, m, l


def _gat_backward(g, z, a_src, a_dst, m, l, out, graph: LoopGraph, slope: float, p_drop: float, seed: int,
                  dz_out: Optional[torch.Tensor] = None):
    """``(dz, da_src, da_dst)`` of the fused forward; ``da_*`` fp32.  ``dz_out``: a row-major [N, H*C] view (any
    leading dimension, e.g. the first columns of a wider gradient) that receives dz instead of a new tensor."""
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
        _lib.check(lib.gmlm_gat_bwd_edges(_ptr(fwd.rowptr), _ptr(fwd.col), n, _ptr(z), _dtype_code(z, "gat"), _ld(z),
                                          _ptr(g), _ld(g), _ptr(a_src), _ptr(a_dst), _ptr(m), _ptr(l), _ptr(t), heads,
                                          head_dim, slope, p_drop, seed, *_hub_args(fwd), _ptr(ws),
                                          ws_bytes, _ptr(alpha_eff), _ptr(d_score), _ptr(da_dst), _stream(dev)),
                   "gat_bwd_edges")
        da_src = torch.empty((a_src.size(0), heads), dtype=torch.float32, device=dev)
        _lib.check(lib.gmlm_segment_sum_f32(_ptr(d_score), _ptr(graph.t2f), _ptr(graph.bwd.rowptr), a_src.size(0),
                                            heads, _ptr(da_src), _stream(dev)), "segment_sum")
    bwd_w = _with_w(graph.bwd, alpha_eff[graph.t2f].contiguous())
    if dz_out is None:
        dz = spmm(g, bwd_w, _lib.AGG_WEIGHTED)
    else:
        dz = _spmm_into(g, bwd_w, dz_out)
    return dz, da_src, da_dst


def _spmm_into(x: torch.Tensor, csr: CSR, out: torch.Tensor) -> torch.Tensor:
    """Weighted ``spmm`` written into a row-major view ``out`` with its own leading dimension."""
    lib = _lib.load()
    if out.dim() != 2 or out.stride(1) != 1 or out.shape != (csr.num_rows, x.size(1)) or out.dtype != x.dtype:
        raise _lib.GmlmError("gat: the dz view must be a row-major [num_rows, H*C] tensor of g's dtype")
    dev = x.device
    feat = int(x.size(1))
    w_heads = int(csr.w.size(1)) if csr.w.dim() == 2 else 1
    n_hub = int(csr.hub_row.numel()) if csr.hub_row is not None else 0
    n_chunks = int(csr.chunk_beg.numel()) if csr.chunk_beg is not None else 0
    n_groups = int(csr.grp_row.numel()) - 1 if csr.grp_row is not None else 0
    mode = _lib.AGG_WEIGHTED if csr.col.numel() else _lib.AGG_SUM      # no edges: every row is zero
    with torch.cuda.device(dev):
        hub_ws = torch.empty(n_chunks * feat, dtype=torch.float32, device=dev) if n_hub else None
        _lib.check(lib.gmlm_spmm_csr(_ptr(x), _dtype_code(x, "spmm_csr"), feat, _ld(x), _ptr(csr.rowptr),
                                     _ptr(csr.col), _ptr(csr.w) if mode == _lib.AGG_WEIGHTED else None,
                                     w_heads if mode == _lib.AGG_WEIGHTED else 1, csr.num_rows, mode, _ptr(csr.grp_row),
                                     n_groups, csr.hub_thresh, n_hub, n_chunks, _ptr(csr.hub_row),
                                     _ptr(csr.hub_chunk_ptr), _ptr(csr.chunk_beg), _ptr(csr.chunk_end), _ptr(hub_ws),
                                     _ptr(out), _ld(out), _stream(dev)), "spmm_csr")
    return out


class _GATAggregate(torch.autograd.Function):
    """Fused edge-softmax aggregation (csrc/gat_fused.cu): one pass, online softmax, alpha never stored."""

    @staticmethod
    def forward(ctx, z, a_src, a_dst, graph: LoopGraph, slope: float, p_drop: float, seed: int):
        z = _rowmajor(z)
        a_src32, a_dst32 = a_src.detach().float().contiguous(), a_dst.detach().float().contiguous()
        out, m, l = _gat_forward(z, a_src32, a_dst32, graph, slope, p_drop, seed)
        ctx.graph, ctx.slope, ctx.p_drop, ctx.seed = graph, float(slope), float(p_drop), int(seed)
        ctx.save_for_backward(z, a_src32, a_dst32, m, l, out)
        ctx.in_dtypes = (a_src.dtype, a_dst.dtype)
        return out

    @staticmethod
    def backward(ctx, g):
        z, a_src, a_dst, m, l, out = ctx.saved_tensors
        g = _rowmajor(g)
        if g.dtype != z.dtype:
            g = g.to(z.dtype)
        dz, da_src, da_dst = _gat_backward(g, z, a_src, a_dst, m, l, out, ctx.graph, ctx.slope, ctx.p_drop, ctx.seed)
        return dz, da_src.to(ctx.in_dtypes[0]), da_dst.to(ctx.in_dtypes[1]), None, None, None, None


class _GATAggregateScored(torch.autograd.Function):
    """The aggregation fed by ONE projection ``y = x @ [W ; w_src ; w_dst]^T`` (``gat_score_weight``):
    ``z = y[:, :H*C]`` is read in place (leading dimension = y's), ``a_src`` / ``a_dst`` are y's next 2H columns.
    The backward writes dz, da_src and da_dst straight into the columns of one gradient buffer shaped like y, so
    nothing assembles the GEMM's output gradient in a separate pass."""

    @staticmethod
    def forward(ctx, y, heads: int, graph: LoopGraph, slope: float, p_drop: float, seed: int):
        y = _rowmajor(y)
        hc = y.size(1) - 2 * heads
        z = y[:, :hc]
        a_src32 = y[:, hc:hc + heads].contiguous()
        a_dst32 = y[:, hc + heads:].contiguous()
        out, m, l = _gat_forward(z, a_src32, a_dst32, graph, slope, p_drop, seed)
        ctx.graph, ctx.slope, ctx.p_drop, ctx.seed, ctx.heads = graph, float(slope), float(p_drop), int(seed), heads
        ctx.save_for_backward(y, a_src32, a_dst32, m, l, out)
        return out

    @staticmethod
    def backward(ctx, g):
        y, a_src, a_dst, m, l, out = ctx.saved_tensors
        heads = ctx.heads
        hc = y.size(1) - 2 * heads
        g = _rowmajor(g)
        if g.dtype != y.dtype:
            g = g.to(y.dtype)
        n, width = y.shape
        per = 4                                   # fp32: 16-byte row pitch, as the GEMM lays out y
        dy = torch.empty((n, (width + per - 1) // per * per), dtype=y.dtype, device=y.device)[:, :width]
        _, da_src, da_dst = _gat_backward(g, y[:, :hc], a_src, a_dst, m, l, out, ctx.graph, ctx.slope, ctx.p_drop,
                                          ctx.seed, dz_out=dy[:, :hc])
        dy[:, hc:hc + heads].copy_(da_src)
        dy[:, hc + heads:].copy_(da_dst)
        return dy, None, None, None, None, None


def gat_aggregate(z, a_src, a_dst, graph: LoopGraph, negative_slope: float = 0.2, dropout: float = 0.0,
                  seed: int = 0) -> torch.Tensor:
    """``out[i,h,:] = sum_j softmax_j(leaky_relu(a_src[j,h] + a_dst[i,h])) * z[j,h,:]`` over the in-edges, with
    optional attention dropout (keep mask = counter-based hash of (seed, edge, head): see ``gat_dropout_mask``)."""
    _require_cuda(z, "z")
    return _GATAggregate.apply(z, a_src, a_dst, graph, negative_slope, dropout, seed)


def gat_score_weight(weight: torch.Tensor, att_src: torch.Tensor, att_dst: torch.Tensor) -> torch.Tensor:
    """``[W ; w_src ; w_dst]`` [H*C + 2H, K]: the projection weight with the attention vectors folded in, so that
    ``x @ W_ext^T = [z | a_src | a_dst]`` with ``a_src[i,h] = sum_c z[i,h,c] att_src[h,c]`` (and ``a_dst`` likewise),
    because ``a_src[i,h] = x_i . (sum_c att_src[h,c] W[h*C+c, :])``.  Differentiable in all three parameters."""
    heads, c = att_src.shape[-2], att_src.shape[-1]
    wv = weight.view(heads, c, weight.size(1))
    w_src = torch.einsum("hc,hck->hk", att_src.reshape(heads, c), wv)
    w_dst = torch.einsum("hc,hck->hk", att_dst.reshape(heads, c), wv)
    return torch.cat([weight, w_src, w_dst], dim=0)


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
    mode).  Row A9 / BASELINE configs[2].  The edge-softmax and the aggregation are ONE kernel pass."""

    def __init__(self, in_channels: int, out_channels: int, heads: int = 1, concat: bool = True,
                 negative_slope: float = 0.2, dropout: float = 0.0, bias: bool = True):
        super().__init__()
        if not 0.0 <= dropout < 1.0:
            raise ValueError("gmlm_b200.GATConv: dropout must be in [0, 1)")
        self.in_channels, self.out_channels, self.heads, self.concat = in_channels, out_channels, heads, concat
        self.negative_slope = negative_slope
        self.dropout = dropout
        self.lin = nn.Linear(in_channels, heads * out_channels, bias=False)
        self.att_src = nn.Parameter(torch.empty(1, heads, out_channels))
        self.att_dst = nn.Parameter(torch.empty(1, heads, out_channels))
        if bias:
            self.bias = nn.Parameter(torch.zeros(heads * out_channels if concat else out_channels))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        glorot_(self.lin.weight)
        glorot_(self.att_src)
        glorot_(self.att_dst)
        if self.bias is not None:
            nn.init.zeros_(self.bias)

    def forward(self, x: torch.Tensor, edge_index, dropout_seed: Optional[int] = None) -> torch.Tensor:
        n, h, c = x.size(0), self.heads, self.out_channels
        graph = edge_index if isinstance(edge_index, LoopGraph) else get_loop_graph(edge_index, n)
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
                out = _GATAggregateScored.apply(y, h, graph, self.negative_slope, p, seed)
        else:
            z = self.lin(x)
            zv = z.view(n, h, c)
            a_src = (zv * self.att_src).sum(-1)
            a_dst = (zv * self.att_dst).sum(-1)
            out = gat_aggregate(z, a_src, a_dst, graph, self.negative_slope, p, seed)
        if not self.concat:
            out = out.view(n, h, c).mean(dim=1)
        return out + self.bias if self.bias is not None else out
