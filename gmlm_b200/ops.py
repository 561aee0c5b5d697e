"""Thin torch layer over the C ABI: tensor checks, output allocation from the caching
allocator, launch on the current stream, autograd registration.

Registered ops (``torch.ops.gmlm.*``, CUDA only — calling them with CPU tensors raises from
the dispatcher; there is no fallback), every one with a fake (meta) implementation:

    degree_i32, edge_type_bucket, csr_build, spmm_csr, colstats, gemm_nt, graphnorm_bwd, layernorm_bwd, soft_mask_bwd
    rgcn_aggregate, plan_aggregate, graphnorm_fwd, layernorm_fwd, soft_mask_fwd      <- differentiable
                                                       (torch.library.register_autograd: backward = the ops above)

Thin functional wrappers used by the modules in ``gmlm_b200.nn``:

    rgcn_aggregate(x, graph)            A5 forward / A14 backward
    graph_norm(x, weight, bias, mean_scale, eps, fuse_gelu)   A7
    soft_mask(x, mask, token, beta)     A11
    layer_norm(x, weight, bias, eps)    A13 (the LayerNorm closing MultiScaleFusion)
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib
from .graph import CSR, RelGraph, _ptr, _require_cuda, _stream

_DT = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16}


def _dtype_code(t: torch.Tensor, what: str) -> int:
    try:
        return _DT[t.dtype]
    except KeyError:
        raise _lib.GmlmError(f"{what}: dtype {t.dtype} unsupported (float32 and bfloat16 only)") from None


def _rowmajor(t: torch.Tensor) -> torch.Tensor:
    """2-D tensor with unit inner stride (a leading dimension is fine, anything else is copied)."""
    if t.dim() != 2:
        raise _lib.GmlmError(f"expected a 2-D tensor, got shape {tuple(t.shape)}")
    if t.size(1) > 0 and t.stride(1) != 1 or (t.size(0) > 1 and t.stride(0) < t.size(1)):
        t = t.contiguous()
    return t


def _ld(t: torch.Tensor) -> int:
    return int(t.stride(0)) if t.size(0) > 1 else int(t.size(1))


_LIB = torch.library.Library("gmlm", "DEF")
_LIB.define("degree_i32(Tensor index, int num_nodes) -> Tensor")
_LIB.define("edge_type_bucket(Tensor src, Tensor deg, int[] bounds) -> Tensor")
_LIB.define("spmm_csr(Tensor x, Tensor rowptr, Tensor col, Tensor? w, int num_rows, int mode, Tensor? grp_row, "
            "int hub_thresh, Tensor? hub_row, Tensor? hub_chunk_ptr, Tensor? chunk_beg, Tensor? chunk_end, "
            "Tensor? hub_col=None, Tensor? hub_w=None, Tensor? band_plan=None) -> Tensor")
_LIB.define("colstats(Tensor x) -> (Tensor, Tensor)")
_LIB.define("graphnorm_fwd(Tensor x, Tensor weight, Tensor bias, Tensor mean_scale, float eps, bool fuse_gelu) "
            "-> (Tensor, Tensor, Tensor)")
_LIB.define("graphnorm_bwd(Tensor x, Tensor gy, Tensor mean, Tensor rstd, Tensor weight, Tensor bias, "
            "Tensor mean_scale, bool fuse_gelu, bool need_gx) -> (Tensor, Tensor, Tensor, Tensor)")
_LIB.define("layernorm_fwd(Tensor x, Tensor weight, Tensor bias, float eps) -> (Tensor, Tensor, Tensor)")
_LIB.define("layernorm_bwd(Tensor x, Tensor gy, Tensor mean, Tensor rstd, Tensor weight, bool need_gx) "
            "-> (Tensor, Tensor, Tensor)")
_LIB.define("soft_mask_fwd(Tensor x, Tensor mask, Tensor token, float beta) -> Tensor")
_LIB.define("soft_mask_bwd(Tensor gy, Tensor mask, float beta, bool need_gx) -> (Tensor, Tensor)")
# differentiable ops (autograd registered below with torch.library.register_autograd)
# a CSR travels as eleven (optional) tensors: rowptr, col, w, grp_row, hub_row, hub_chunk_ptr, chunk_beg, chunk_end,
# hub_col, hub_w, band_plan
_CSR_ARGS = ("Tensor {p}rowptr, Tensor {p}col, Tensor? {p}w, Tensor? {p}grp, Tensor? {p}hub_row, "
             "Tensor? {p}hub_chunk_ptr, Tensor? {p}chunk_beg, Tensor? {p}chunk_end, Tensor? {p}hub_col, "
             "Tensor? {p}hub_w, Tensor? {p}band_plan")
_NC = 11
_LIB.define("rgcn_aggregate(Tensor x, " + _CSR_ARGS.format(p="f_") + ", " + _CSR_ARGS.format(p="b_") +
            ", int[] meta) -> Tensor")
_LIB.define("plan_aggregate(Tensor rows, " + _CSR_ARGS.format(p="f_") + ", " + _CSR_ARGS.format(p="b_") +
            ", int[] meta) -> Tensor")
_LIB.define("gemm_nt(Tensor a1, Tensor b, Tensor? bias, Tensor? a2, ScalarType out_dtype) -> Tensor")
_LIB.define("csr_build(Tensor row, Tensor col, Tensor? rel, Tensor? keep, int num_rows, int num_cols, int num_relations, "
            "int[] slot_of_rel, int num_slots) -> (Tensor, Tensor, Tensor, Tensor)")


# ------------------------------------------------------------------------------ A1 / A2
def _degree_i32(index: torch.Tensor, num_nodes: int) -> torch.Tensor:
    lib = _lib.load()
    index = index.reshape(-1).contiguous()
    if index.dtype != torch.int64:
        index = index.long()
    with torch.cuda.device(index.device):
        deg = torch.empty(num_nodes, dtype=torch.int32, device=index.device)
        _lib.check(lib.gmlm_degree_i32(_ptr(index), index.numel(), num_nodes, _ptr(deg), 0, _stream(index.device)),
                   "degree")
    return deg


def _edge_type_bucket(src: torch.Tensor, deg: torch.Tensor, bounds: Sequence[int]) -> torch.Tensor:
    lib = _lib.load()
    src = src.reshape(-1).contiguous()
    if src.dtype != torch.int64:
        src = src.long()
    nb = len(bounds)
    arr = (C.c_int32 * max(nb, 1))(*[int(b) for b in bounds])
    with torch.cuda.device(src.device):
        out = torch.empty(src.numel(), dtype=torch.int64, device=src.device)
        _lib.check(lib.gmlm_edge_type_bucket(_ptr(src), src.numel(), _ptr(deg), deg.numel(), arr, nb, _ptr(out),
                                             _stream(src.device)), "edge_type_bucket")
    return out


# ------------------------------------------------------------------------------ A5 / A14
def _spmm_csr(x: torch.Tensor, csr: CSR, mode: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The aggregation kernel: out[r] = reduce over row r of ``csr`` (``mode`` AGG_SUM / AGG_MEAN / AGG_WEIGHTED; the
    weighted mode reads ``csr.w``, one column per head when 2-D, and ``csr.hub_w`` for the band-ordered hub chunks).
    ``out``: a row-major [num_rows, F] tensor of x's dtype, any leading dimension, written in place."""
    lib = _lib.load()
    x = _rowmajor(x)
    feat = int(x.size(1))
    dev = x.device
    w, hub_w = (csr.w, csr.hub_w) if mode == _lib.AGG_WEIGHTED else (None, None)
    n_hub = int(csr.hub_row.numel()) if csr.hub_row is not None else 0
    n_chunks = int(csr.chunk_beg.numel()) if csr.chunk_beg is not None else 0
    n_groups = int(csr.grp_row.numel()) - 1 if csr.grp_row is not None else 0
    n_band = (int(csr.band_plan.numel()) - n_hub - 2) // 2 if (csr.band_plan is not None and n_hub) else 0
    w_heads = int(w.size(1)) if (w is not None and w.dim() == 2) else 1
    if csr.col.numel() == 0 and mode == _lib.AGG_WEIGHTED:
        mode, w, w_heads = _lib.AGG_SUM, None, 1          # no edges: every row is empty, the result is zeros
    with torch.cuda.device(dev):
        if out is None:
            out = torch.empty((csr.num_rows, feat), dtype=x.dtype, device=dev)
        elif out.dim() != 2 or out.stride(1) != 1 or out.shape != (csr.num_rows, feat) or out.dtype != x.dtype:
            raise _lib.GmlmError("spmm: `out` must be a row-major [num_rows, feat] tensor of x's dtype")
        hub_ws = torch.empty(max(n_chunks, n_band) * feat, dtype=torch.float32, device=dev) if n_hub else None
        _lib.check(lib.gmlm_spmm_csr_banded(_ptr(x), _dtype_code(x, "spmm_csr"), feat, _ld(x), _ptr(csr.rowptr),
                                            _ptr(csr.col), _ptr(w), w_heads, csr.num_rows, mode, _ptr(csr.grp_row),
                                            n_groups, csr.hub_thresh, n_hub, n_chunks, _ptr(csr.hub_row),
                                            _ptr(csr.hub_chunk_ptr), _ptr(csr.chunk_beg), _ptr(csr.chunk_end), n_band,
                                            _ptr(csr.band_plan if n_band else None), _ptr(csr.hub_col), _ptr(hub_w),
                                            _ptr(hub_ws), _ptr(out), _ld(out), _stream(dev)), "spmm_csr")
    return out


def spmm(x: torch.Tensor, csr: CSR, mode: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[r] = reduce over row r of csr (no autograd).  ``out`` lets the result land in a caller-owned
    buffer (e.g. NVLink-peer-visible symmetric memory for the halo exchange)."""
    _require_cuda(x, "x")
    if out is not None:
        return _spmm_csr(x, csr, mode, out)
    c, (rows, thresh) = csr_pack(csr)
    return _spmm_op(x, c, rows, thresh, mode)


def _spmm_csr_op(x, rowptr, col, w, num_rows, mode, grp_row, hub_thresh, hub_row, hub_chunk_ptr, chunk_beg, chunk_end,
                 hub_col=None, hub_w=None, band_plan=None):
    c = [rowptr, col, w, grp_row, hub_row, hub_chunk_ptr, chunk_beg, chunk_end, hub_col, hub_w, band_plan]
    return _spmm_csr(x, _csr_unpack(c, num_rows, hub_thresh), mode)


# ------------------------------------------------------------------------------ A7
def _colstats(x: torch.Tensor):
    lib = _lib.load()
    x = _rowmajor(x)
    n, c = x.shape
    dev = x.device
    with torch.cuda.device(dev):
        colsum = torch.empty(c, dtype=torch.float64, device=dev)
        colsq = torch.empty(c, dtype=torch.float64, device=dev)
        ws_bytes = lib.gmlm_colstats_workspace_bytes(n, c)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.check(lib.gmlm_colstats(_ptr(x), _dtype_code(x, "colstats"), n, c, _ld(x), _ptr(colsum), _ptr(colsq),
                                     _ptr(ws), ws_bytes, _stream(dev)), "colstats")
    return colsum, colsq


def _f32c(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.float32).contiguous()


def graphnorm_apply_stats(x, colsum, colsq, weight, bias, mean_scale, eps, fuse_gelu, stat_rows=0):
    """Normalise pass of A7 given the fp64 column sums; ``stat_rows`` = rows the sums cover (0 = x's rows;
    the whole-graph count when x holds one rank's rows of a partition)."""
    lib = _lib.load()
    x = _rowmajor(x)
    n, c = x.shape
    dev = x.device
    weight, bias, mean_scale = _f32c(weight), _f32c(bias), _f32c(mean_scale)
    with torch.cuda.device(dev):
        y = torch.empty((n, c), dtype=x.dtype, device=dev)
        mean = torch.empty(c, dtype=torch.float32, device=dev)
        rstd = torch.empty(c, dtype=torch.float32, device=dev)
        _lib.check(lib.gmlm_graphnorm_fwd(_ptr(x), _dtype_code(x, "graphnorm"), n, c, _ld(x), _ptr(colsum),
                                          _ptr(colsq), _ptr(weight), _ptr(bias), _ptr(mean_scale), float(eps),
                                          int(bool(fuse_gelu)), _ptr(y), c, _ptr(mean), _ptr(rstd), int(stat_rows),
                                          _stream(dev)), "graphnorm_fwd")
    return y, mean, rstd


def graphnorm_bwd_stats(x, gy, mean, rstd, weight, bias, mean_scale, fuse_gelu):
    """Column sums the backward needs (sum dn, sum dn*xhat), fp64, local rows only."""
    lib = _lib.load()
    x = _rowmajor(x)
    gy = _rowmajor(gy)
    if gy.dtype != x.dtype:
        gy = gy.to(x.dtype)
    n, c = x.shape
    dev = x.device
    weight, bias, mean_scale = _f32c(weight), _f32c(bias), _f32c(mean_scale)
    with torch.cuda.device(dev):
        s1 = torch.empty(c, dtype=torch.float64, device=dev)
        s2 = torch.empty(c, dtype=torch.float64, device=dev)
        ws_bytes = lib.gmlm_colstats_workspace_bytes(n, c)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.check(lib.gmlm_graphnorm_bwd_stats(_ptr(x), _ptr(gy), _dtype_code(x, "graphnorm_bwd"), n, c, _ld(x),
                                                _ld(gy), _ptr(mean), _ptr(rstd), _ptr(weight), _ptr(bias),
                                                _ptr(mean_scale), int(bool(fuse_gelu)), _ptr(s1), _ptr(s2), _ptr(ws),
                                                ws_bytes, _stream(dev)), "graphnorm_bwd_stats")
    return s1, s2


def graphnorm_bwd_apply(x, gy, mean, rstd, weight, bias, mean_scale, fuse_gelu, s1, s2, need_gx, stat_rows=0):
    lib = _lib.load()
    x = _rowmajor(x)
    gy = _rowmajor(gy)
    if gy.dtype != x.dtype:
        gy = gy.to(x.dtype)
    n, c = x.shape
    dev = x.device
    weight, bias, mean_scale = _f32c(weight), _f32c(bias), _f32c(mean_scale)
    with torch.cuda.device(dev):
        gx = torch.empty((n, c), dtype=x.dtype, device=dev) if need_gx else torch.empty(0, dtype=x.dtype, device=dev)
        gw = torch.empty(c, dtype=torch.float32, device=dev)
        gb = torch.empty(c, dtype=torch.float32, device=dev)
        gms = torch.empty(c, dtype=torch.float32, device=dev)
        _lib.check(lib.gmlm_graphnorm_bwd_apply(_ptr(x), _ptr(gy), _dtype_code(x, "graphnorm_bwd"), n, c, _ld(x),
                                                _ld(gy), _ptr(mean), _ptr(rstd), _ptr(weight), _ptr(bias),
                                                _ptr(mean_scale), int(bool(fuse_gelu)), _ptr(s1), _ptr(s2),
                                                _ptr(gx) if need_gx else C.c_void_p(0), c, _ptr(gw), _ptr(gb),
                                                _ptr(gms), int(stat_rows), _stream(dev)), "graphnorm_bwd_apply")
    return gx, gw, gb, gms


def _graphnorm_fwd(x, weight, bias, mean_scale, eps, fuse_gelu):
    colsum, colsq = _colstats(x)
    return graphnorm_apply_stats(x, colsum, colsq, weight, bias, mean_scale, eps, fuse_gelu)


def _graphnorm_bwd(x, gy, mean, rstd, weight, bias, mean_scale, fuse_gelu, need_gx):
    s1, s2 = graphnorm_bwd_stats(x, gy, mean, rstd, weight, bias, mean_scale, fuse_gelu)
    return graphnorm_bwd_apply(x, gy, mean, rstd, weight, bias, mean_scale, fuse_gelu, s1, s2, need_gx)


# ------------------------------------------------------------------------------ A13 LayerNorm
def layer_norm_ok(x: torch.Tensor) -> bool:
    """Shapes the row-wise kernel takes: CUDA fp32/bf16 [N, C], C a multiple of the 16-byte pack, C <= 1024.
    Any strides and storage offset: a view the kernel cannot read in 16-byte packs is copied first."""
    if not (x.is_cuda and x.dim() == 2 and x.dtype in _DT and x.size(0) >= 1):
        return False
    vec = 4 if x.dtype == torch.float32 else 8
    return x.size(1) % vec == 0 and 0 < x.size(1) <= _lib.load().gmlm_layernorm_max_channels(_DT[x.dtype])


def _packed_rows(t: torch.Tensor) -> torch.Tensor:
    """``_rowmajor`` plus what the LayerNorm kernel reads in 16-byte packs: a 16-byte aligned base and a leading
    dimension that is a whole number of packs.  A view that lacks either (a column slice at an odd offset, the
    gradient autograd hands back for one block of a ``torch.cat``) is copied."""
    t = _rowmajor(t)
    vec = 16 // t.element_size()
    if t.data_ptr() % 16 or _ld(t) % vec:
        t = t.clone(memory_format=torch.contiguous_format)
    return t


def _layernorm_fwd(x, weight, bias, eps):
    lib = _lib.load()
    x = _packed_rows(x)
    n, c = x.shape
    dev = x.device
    weight, bias = _f32c(weight), _f32c(bias)
    with torch.cuda.device(dev):
        y = torch.empty((n, c), dtype=x.dtype, device=dev)
        mean = torch.empty(n, dtype=torch.float32, device=dev)
        rstd = torch.empty(n, dtype=torch.float32, device=dev)
        _lib.check(lib.gmlm_layernorm_fwd(_ptr(x), _dtype_code(x, "layernorm"), n, c, _ld(x), _ptr(weight), _ptr(bias),
                                          float(eps), _ptr(y), c, _ptr(mean), _ptr(rstd), _stream(dev)),
                   "layernorm_fwd")
    return y, mean, rstd


def _layernorm_bwd(x, gy, mean, rstd, weight, need_gx):
    lib = _lib.load()
    x = _packed_rows(x)
    if gy.dtype != x.dtype:
        gy = gy.to(x.dtype)
    gy = _packed_rows(gy)
    n, c = x.shape
    dev = x.device
    weight = _f32c(weight)
    with torch.cuda.device(dev):
        gx = torch.empty((n, c), dtype=x.dtype, device=dev) if need_gx else torch.empty(0, dtype=x.dtype, device=dev)
        gw = torch.empty(c, dtype=torch.float32, device=dev)
        gb = torch.empty(c, dtype=torch.float32, device=dev)
        ws_bytes = lib.gmlm_layernorm_bwd_workspace_bytes(n, c)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.check(lib.gmlm_layernorm_bwd(_ptr(x), _ptr(gy), _dtype_code(x, "layernorm_bwd"), n, c, _ld(x), _ld(gy),
                                          _ptr(weight), _ptr(mean), _ptr(rstd),
                                          _ptr(gx) if need_gx else C.c_void_p(0), c, _ptr(gw), _ptr(gb), _ptr(ws),
                                          ws_bytes, _stream(dev)), "layernorm_bwd")
    return gx, gw, gb


# ------------------------------------------------------------------------------ A11
def _mask_u8(mask: torch.Tensor, n: int) -> torch.Tensor:
    mask = mask.reshape(-1)
    if mask.numel() != n:
        raise _lib.GmlmError(f"mask has {mask.numel()} entries for {n} rows")
    if mask.dtype == torch.bool:
        return mask.contiguous().view(torch.uint8)
    return (mask != 0).view(torch.uint8)


def _soft_mask_fwd(x, mask, token, beta):
    lib = _lib.load()
    x = _rowmajor(x)
    n, f = x.shape
    dev = x.device
    m = _mask_u8(mask.to(dev), n)
    token = _f32c(token.to(dev)).reshape(-1)
    if token.numel() != f:
        raise _lib.GmlmError(f"mask token has {token.numel()} features, x has {f}")
    with torch.cuda.device(dev):
        y = torch.empty((n, f), dtype=x.dtype, device=dev)
        _lib.check(lib.gmlm_soft_mask_fwd(_ptr(x), _dtype_code(x, "soft_mask"), n, f, _ld(x), _ptr(m), _ptr(token),
                                          float(beta), _ptr(y), f, _stream(dev)), "soft_mask_fwd")
    return y


def _soft_mask_bwd(gy, mask, beta, need_gx):
    lib = _lib.load()
    gy = _rowmajor(gy)
    n, f = gy.shape
    dev = gy.device
    m = _mask_u8(mask.to(dev), n)
    with torch.cuda.device(dev):
        g_token = torch.empty(f, dtype=torch.float32, device=dev)
        gx = torch.empty((n, f), dtype=gy.dtype, device=dev) if need_gx else torch.empty(0, dtype=gy.dtype, device=dev)
        ws_bytes = lib.gmlm_soft_mask_bwd_workspace_bytes(n, f)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.check(lib.gmlm_soft_mask_bwd(_ptr(gy), _dtype_code(gy, "soft_mask_bwd"), n, f, _ld(gy), _ptr(m),
                                          float(beta), _ptr(g_token), _ptr(gx) if need_gx else C.c_void_p(0), f,
                                          _ptr(ws), ws_bytes, _stream(dev)), "soft_mask_bwd")
    return g_token, gx


_LIB.impl("degree_i32", _degree_i32, "CUDA")
_LIB.impl("edge_type_bucket", _edge_type_bucket, "CUDA")
_LIB.impl("spmm_csr", _spmm_csr_op, "CUDA")
_LIB.impl("colstats", _colstats, "CUDA")
_LIB.impl("graphnorm_fwd", _graphnorm_fwd, "CUDA")
_LIB.impl("graphnorm_bwd", _graphnorm_bwd, "CUDA")
_LIB.impl("layernorm_fwd", _layernorm_fwd, "CUDA")
_LIB.impl("layernorm_bwd", _layernorm_bwd, "CUDA")
_LIB.impl("soft_mask_fwd", _soft_mask_fwd, "CUDA")
_LIB.impl("soft_mask_bwd", _soft_mask_bwd, "CUDA")


# ------------------------------------------------------------------------------ differentiable custom ops
# torch.ops.gmlm.{rgcn_aggregate, plan_aggregate, graphnorm_fwd, layernorm_fwd, soft_mask_fwd} carry their
# backward (torch.library.register_autograd) and a fake implementation (register_fake), so they can be called,
# traced and differentiated as ordinary torch operators; the thin functions further down only validate arguments.
def csr_pack(csr: CSR):
    """CSR -> (Tensor?[11], [num_rows, hub_thresh]): rowptr, col, w, grp_row, hub_row, hub_chunk_ptr, chunk_beg,
    chunk_end, hub_col, hub_w, band_plan."""
    return ([csr.rowptr, csr.col, csr.w, csr.grp_row, csr.hub_row, csr.hub_chunk_ptr, csr.chunk_beg, csr.chunk_end,
             csr.hub_col, csr.hub_w, csr.band_plan], [int(csr.num_rows), int(csr.hub_thresh)])


def _csr_unpack(c, num_rows: int, hub_thresh: int) -> CSR:
    """The CSR of ``csr_pack``'s eleven tensors (the fields the aggregation kernel reads)."""
    rowptr, col, w, grp_row, hub_row, hub_chunk_ptr, chunk_beg, chunk_end, hub_col, hub_w, band_plan = c
    return CSR(rowptr=rowptr, col=col, num_rows=num_rows, w=w, hub_thresh=hub_thresh, hub_row=hub_row,
               hub_chunk_ptr=hub_chunk_ptr, chunk_beg=chunk_beg, chunk_end=chunk_end, hub_col=hub_col, hub_w=hub_w,
               band_plan=band_plan, grp_row=grp_row)


def _spmm_op(x, c, rows: int, thresh: int, mode: int):
    """``torch.ops.gmlm.spmm_csr`` on a CSR packed by ``csr_pack``."""
    return torch.ops.gmlm.spmm_csr(x, c[0], c[1], c[2], rows, mode, c[3], thresh, *c[4:])


def _rgcn_aggregate_impl(x, *a):
    fwd, meta = a[0:_NC], a[2 * _NC]
    rows_f, thresh_f, _, _, n_nodes, n_slots = meta
    h = _spmm_csr(x, _csr_unpack(fwd, rows_f, thresh_f), _lib.AGG_MEAN)     # [N*S, F]
    return h.view(n_nodes, n_slots * x.size(1))


def _plan_aggregate_impl(rows, *a):
    fwd, meta = a[0:_NC], a[2 * _NC]
    return _spmm_csr(rows, _csr_unpack(fwd, meta[0], meta[1]), _lib.AGG_WEIGHTED)


def _gemm_nt_op(a1, b, bias, a2, out_dtype):
    return gemm_nt(a1, b, bias=bias, a2=a2, out_dtype=out_dtype).contiguous()


def _csr_build_op(row, col, rel, keep, num_rows, num_cols, num_relations, slot_of_rel, num_slots):
    """(rowptr int32 [num_rows*num_slots+1], col int32 [E], perm int32 [E], seg_of_edge int32 [E]) of the CSR keyed
    on ``row*num_slots + slot_of_rel[rel]`` (stable: original edge order inside a segment); A3.  ``keep`` (uint8 /
    bool [E], optional) is an edge-dropout mask fused into the build: only the first rowptr[-1] entries of col / perm
    are then the CSR."""
    lib = _lib.load()
    dev = row.device
    E = int(row.numel())
    row, col = row.contiguous(), col.contiguous()
    rel = rel.contiguous() if rel is not None else None
    rows_total = num_rows * num_slots
    with torch.cuda.device(dev):
        rowptr = torch.empty(rows_total + 1, dtype=torch.int32, device=dev)
        colv = torch.empty(E, dtype=torch.int32, device=dev)
        perm = torch.empty(E, dtype=torch.int32, device=dev)
        seg = torch.empty(E, dtype=torch.int32, device=dev)
        ws_bytes = lib.gmlm_csr_workspace_bytes(max(E, 1), rows_total)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        slots = (C.c_int32 * max(num_relations, 1))(*[int(v) for v in slot_of_rel]) if rel is not None else None
        keep_u8 = _mask_u8(keep, E) if keep is not None else None
        nnz = C.c_int64(0)
        # csr_build keys on `dst`; here the CSR row plays that role and `col` is the gathered id
        _lib.check(lib.gmlm_csr_build(_ptr(col), _ptr(row), _ptr(rel), _ptr(keep_u8), E, num_rows, num_cols,
                                      num_relations, slots, num_slots, _ptr(rowptr), _ptr(colv), _ptr(perm), _ptr(seg),
                                      C.byref(nnz) if keep is not None else None, _ptr(ws), ws_bytes, _stream(dev)),
                   "csr_build")
    return rowptr, colv, perm, seg


_LIB.impl("rgcn_aggregate", _rgcn_aggregate_impl, "CUDA")
_LIB.impl("plan_aggregate", _plan_aggregate_impl, "CUDA")
_LIB.impl("gemm_nt", _gemm_nt_op, "CUDA")
_LIB.impl("csr_build", _csr_build_op, "CUDA")


# ---- fake (meta) implementations: shapes and dtypes only
@torch.library.register_fake("gmlm::degree_i32")
def _(index, num_nodes):
    return index.new_empty((num_nodes,), dtype=torch.int32)


@torch.library.register_fake("gmlm::edge_type_bucket")
def _(src, deg, bounds):
    return src.new_empty((src.numel(),), dtype=torch.int64)


@torch.library.register_fake("gmlm::spmm_csr")
def _(x, rowptr, col, w, num_rows, mode, grp_row, hub_thresh, hub_row, hub_chunk_ptr, chunk_beg, chunk_end,
      hub_col=None, hub_w=None, band_plan=None):
    return x.new_empty((num_rows, x.size(1)))


@torch.library.register_fake("gmlm::colstats")
def _(x):
    return x.new_empty((x.size(1),), dtype=torch.float64), x.new_empty((x.size(1),), dtype=torch.float64)


@torch.library.register_fake("gmlm::graphnorm_fwd")
def _(x, weight, bias, mean_scale, eps, fuse_gelu):
    c = x.size(1)
    return torch.empty_like(x), x.new_empty((c,), dtype=torch.float32), x.new_empty((c,), dtype=torch.float32)


@torch.library.register_fake("gmlm::graphnorm_bwd")
def _(x, gy, mean, rstd, weight, bias, mean_scale, fuse_gelu, need_gx):
    c = x.size(1)
    f = lambda: x.new_empty((c,), dtype=torch.float32)   # noqa: E731
    return (torch.empty_like(x) if need_gx else x.new_empty((0,))), f(), f(), f()


@torch.library.register_fake("gmlm::layernorm_fwd")
def _(x, weight, bias, eps):
    n = x.size(0)
    return torch.empty_like(x), x.new_empty((n,), dtype=torch.float32), x.new_empty((n,), dtype=torch.float32)


@torch.library.register_fake("gmlm::layernorm_bwd")
def _(x, gy, mean, rstd, weight, need_gx):
    c = x.size(1)
    return ((torch.empty_like(x) if need_gx else x.new_empty((0,))), x.new_empty((c,), dtype=torch.float32),
            x.new_empty((c,), dtype=torch.float32))


@torch.library.register_fake("gmlm::soft_mask_fwd")
def _(x, mask, token, beta):
    return torch.empty_like(x)


@torch.library.register_fake("gmlm::soft_mask_bwd")
def _(gy, mask, beta, need_gx):
    return gy.new_empty((gy.size(1),), dtype=torch.float32), (torch.empty_like(gy) if need_gx else gy.new_empty((0,)))


@torch.library.register_fake("gmlm::rgcn_aggregate")
def _(x, *a):
    meta = a[2 * _NC]
    return x.new_empty((meta[4], meta[5] * x.size(1)))


@torch.library.register_fake("gmlm::plan_aggregate")
def _(rows, *a):
    return rows.new_empty((a[2 * _NC][0], rows.size(1)))


@torch.library.register_fake("gmlm::gemm_nt")
def _(a1, b, bias, a2, out_dtype):
    return a1.new_empty((a1.size(0), b.size(0)), dtype=out_dtype)


@torch.library.register_fake("gmlm::csr_build")
def _(row, col, rel, keep, num_rows, num_cols, num_relations, slot_of_rel, num_slots):
    e = row.numel()
    i32 = lambda k: row.new_empty((k,), dtype=torch.int32)   # noqa: E731
    return i32(num_rows * num_slots + 1), i32(e), i32(e), i32(e)


# ---- autograd formulas
def _rgcn_aggregate_setup(ctx, inputs, output):
    x = inputs[0]
    ctx.bwd, ctx.meta, ctx.x_dtype = inputs[1 + _NC:1 + 2 * _NC], inputs[1 + 2 * _NC], x.dtype


def _rgcn_aggregate_backward(ctx, gh):
    _, _, rows_b, thresh_b, n_nodes, n_slots = ctx.meta
    gh = gh.contiguous()
    if gh.dtype != ctx.x_dtype:
        gh = gh.to(ctx.x_dtype)
    feat = gh.size(1) // n_slots
    # A14: gather on the transposed CSR
    gx = _spmm_op(gh.view(n_nodes * n_slots, feat), ctx.bwd, rows_b, thresh_b, _lib.AGG_WEIGHTED)
    return (gx,) + (None,) * (2 * _NC + 1)


def _plan_aggregate_setup(ctx, inputs, output):
    ctx.bwd, ctx.meta, ctx.in_dtype = inputs[1 + _NC:1 + 2 * _NC], inputs[1 + 2 * _NC], inputs[0].dtype


def _plan_aggregate_backward(ctx, g):
    g = g.contiguous()
    if g.dtype != ctx.in_dtype:
        g = g.to(ctx.in_dtype)
    return (_spmm_op(g, ctx.bwd, ctx.meta[2], ctx.meta[3], _lib.AGG_WEIGHTED),) + (None,) * (2 * _NC + 1)


def _graphnorm_setup(ctx, inputs, output):
    x, weight, bias, mean_scale, eps, fuse_gelu = inputs
    _, mean, rstd = output
    ctx.save_for_backward(x, mean, rstd, weight, bias, mean_scale)
    ctx.fuse_gelu = bool(fuse_gelu)


def _graphnorm_backward(ctx, gy, g_mean, g_rstd):
    x, mean, rstd, weight, bias, mean_scale = ctx.saved_tensors
    gx, gw, gb, gms = torch.ops.gmlm.graphnorm_bwd(x, gy, mean, rstd, weight, bias, mean_scale, ctx.fuse_gelu,
                                                   ctx.needs_input_grad[0])
    return (gx if ctx.needs_input_grad[0] else None,
            gw.to(weight.dtype) if ctx.needs_input_grad[1] else None,
            gb.to(bias.dtype) if ctx.needs_input_grad[2] else None,
            gms.to(mean_scale.dtype) if ctx.needs_input_grad[3] else None, None, None)


def _layernorm_setup(ctx, inputs, output):
    x, weight, bias, eps = inputs
    _, mean, rstd = output
    ctx.save_for_backward(x, mean, rstd, weight)
    ctx.bias_dtype = bias.dtype


def _layernorm_backward(ctx, gy, g_mean, g_rstd):
    x, mean, rstd, weight = ctx.saved_tensors
    gx, gw, gb = torch.ops.gmlm.layernorm_bwd(x, gy, mean, rstd, weight, ctx.needs_input_grad[0])
    return (gx if ctx.needs_input_grad[0] else None, gw.to(weight.dtype) if ctx.needs_input_grad[1] else None,
            gb.to(ctx.bias_dtype) if ctx.needs_input_grad[2] else None, None)


def _soft_mask_setup(ctx, inputs, output):
    x, mask, token, beta = inputs
    ctx.save_for_backward(mask)
    ctx.beta, ctx.token_shape, ctx.token_dtype = float(beta), token.shape, token.dtype


def _soft_mask_backward(ctx, gy):
    (mask,) = ctx.saved_tensors
    g_token, gx = torch.ops.gmlm.soft_mask_bwd(gy, mask, ctx.beta, ctx.needs_input_grad[0])
    return (gx if ctx.needs_input_grad[0] else None, None,
            g_token.view(ctx.token_shape).to(ctx.token_dtype) if ctx.needs_input_grad[2] else None, None)


torch.library.register_autograd("gmlm::rgcn_aggregate", _rgcn_aggregate_backward, setup_context=_rgcn_aggregate_setup)
torch.library.register_autograd("gmlm::plan_aggregate", _plan_aggregate_backward, setup_context=_plan_aggregate_setup)
torch.library.register_autograd("gmlm::graphnorm_fwd", _graphnorm_backward, setup_context=_graphnorm_setup)
torch.library.register_autograd("gmlm::layernorm_fwd", _layernorm_backward, setup_context=_layernorm_setup)
torch.library.register_autograd("gmlm::soft_mask_fwd", _soft_mask_backward, setup_context=_soft_mask_setup)


# ------------------------------------------------------------------------------ A6 dense transform (tcgen05)
_OPS16 = (torch.bfloat16, torch.float16)


def _op_code(dt: torch.dtype) -> int:
    return {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16, torch.float16: _lib.F16}[dt]


def _tma_rows(t: torch.Tensor, dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """``t`` [M, K] as a TMA-readable operand of type ``dtype``: unit inner stride, 16-byte aligned rows.  A cast
    and / or a pitch fix is ONE copy into a buffer whose pitch is rounded up to 16 bytes (K = 300 fp16: pitch 304)."""
    dtype = dtype or t.dtype
    es = torch.empty((), dtype=dtype).element_size()
    if (t.dtype == dtype and t.dim() == 2 and t.stride(1) == 1 and (t.stride(0) * es) % 16 == 0
            and t.data_ptr() % 16 == 0 and t.stride(0) >= t.size(1)):
        return t
    m, k = t.shape
    per = 16 // es
    buf = torch.empty((m, (k + per - 1) // per * per), dtype=dtype, device=t.device)
    view = buf[:, :k]
    view.copy_(t)
    return view


def gemm_nt(a1, b: torch.Tensor, bias: Optional[torch.Tensor] = None, a2: Optional[torch.Tensor] = None,
            out_dtype: Optional[torch.dtype] = None, split: int = 0, addend: Optional[torch.Tensor] = None):
    """``[a1 | a2 | ..] @ b.T + bias (+ addend)`` on the tcgen05 tensor cores: bf16 / fp16 operands (fp32 accumulate), or
    fp32 operands as 3xTF32 (hi/lo split in shared memory, three MMAs per k-step: fp32-grade accuracy, 1e-5 gate).

    a1: one [M,K1] tensor or a list of up to four [M,K_i] sources (never concatenated in memory); a2 [M,K2]
    (optional); b [N, sum K], all bf16 (or all fp16) with unit inner stride and a 16-byte row pitch (anything else is
    copied once); any K, N.  Returns C [M,N] (bf16 or fp32), or (C[:, :split], C[:, split:]) as two contiguous tensors
    when ``split`` > 0, or a list of up to four tensors when ``split`` is a list of column widths (more than two:
    multiples of 64).  ``addend`` [M,N] of the output type is added in the epilogue (single output only)."""
    lib = _lib.load()
    srcs = list(a1) if isinstance(a1, (list, tuple)) else [a1]
    if a2 is not None:
        srcs.append(a2)
    _require_cuda(srcs[0], "a1")
    op = srcs[0].dtype
    if op not in _OPS16 + (torch.float32,) or b.dtype != op or any(t.dtype != op for t in srcs):
        raise _lib.GmlmError("gemm_nt: operands must all be bfloat16, all float16 or all float32")
    if not 1 <= len(srcs) <= 4:
        raise _lib.GmlmError("gemm_nt: one to four A sources")
    m = int(srcs[0].size(0))
    if any(t.dim() != 2 or t.size(0) != m for t in srcs) or b.dim() != 2 or b.size(1) != sum(int(t.size(1)) for t in srcs):
        raise _lib.GmlmError(f"gemm_nt: shape mismatch a {[tuple(t.shape) for t in srcs]} b {tuple(b.shape)}")
    if any(t.size(1) % (16 // t.element_size()) for t in srcs[:-1]):
        srcs = [torch.cat(srcs, dim=1)]      # a source must start on a 16-byte column boundary of b: concatenate
    srcs = [_tma_rows(t) for t in srcs]
    b = _tma_rows(b)
    n = int(b.size(0))
    out_dtype = out_dtype or (torch.bfloat16 if op == torch.bfloat16 else torch.float32)
    if out_dtype not in _DT or (op == torch.float32 and out_dtype != torch.float32):
        raise _lib.GmlmError("gemm_nt: output must be float32 or bfloat16 (float32 for float32 operands)")
    per = 16 // torch.empty((), dtype=out_dtype).element_size()
    dev = srcs[0].device
    bias32 = bias.detach().float().contiguous() if bias is not None else None
    if addend is not None:
        if split or addend.shape != (m, n) or addend.dtype != out_dtype:
            raise _lib.GmlmError("gemm_nt: addend must be [M, N] of the output type (single output)")
        addend = _tma_rows(addend)

    def alloc(cols):          # contiguous when the width allows a 16-byte pitch, else a padded buffer's view
        if cols % per == 0:
            return torch.empty((m, cols), dtype=out_dtype, device=dev)
        return torch.empty((m, (cols + per - 1) // per * per), dtype=out_dtype, device=dev)[:, :cols]

    if isinstance(split, (list, tuple)):
        widths = [int(v) for v in split]
        if sum(widths) != n or any(v <= 0 for v in widths) or not 1 <= len(widths) <= 4:
            raise _lib.GmlmError(f"gemm_nt: output widths {widths} do not add up to N = {n}")
        if len(widths) > 2 and any(v % 64 for v in widths[:-1]):
            raise _lib.GmlmError("gemm_nt: more than two outputs must be cut at multiples of 64 columns")
    elif split and 0 < split < n:
        widths = [int(split), n - int(split)]
    else:
        widths = [n]
    if addend is not None and len(widths) > 1:
        raise _lib.GmlmError("gemm_nt: the addend goes with a single output")
    with torch.cuda.device(dev):
        outs = [alloc(v) for v in widths]
        k = len(srcs)
        ptrs = (C.c_void_p * k)(*[t.data_ptr() for t in srcs])
        ldas = (C.c_int64 * k)(*[_ld(t) for t in srcs])
        ks = (C.c_int64 * k)(*[int(t.size(1)) for t in srcs])
        no = len(outs)
        cptrs = (C.c_void_p * no)(*[t.data_ptr() for t in outs])
        ldcs = (C.c_int64 * no)(*[_ld(t) for t in outs])
        ns = (C.c_int64 * no)(*widths)
        _lib.check(lib.gmlm_gemm_nt_multi(k, ptrs, ldas, ks, _ptr(b), _ld(b), _ptr(bias32), _ptr(addend),
                                          _ld(addend) if addend is not None else 0, m, no, cptrs, ldcs, ns,
                                          _op_code(op), _DT[out_dtype], _stream(dev)), "gemm_nt")
    if isinstance(split, (list, tuple)):
        return outs
    return tuple(outs) if len(outs) > 1 else outs[0]


def gemm_tn(srcs, g: torch.Tensor) -> torch.Tensor:
    """``cat(srcs, 1).T @ g`` -> fp32 [sum K_i, N] on the tcgen05 tensor cores: the weight-gradient reduction over all
    rows (dW = H^T g, droot = x^T g in ONE launch over the two sources; dWt = g^T x of the linears).  ``srcs``: one
    to four [M, K_i] tensors, ``g`` [M, N], all bf16 or all fp16; operands are read as they lie (no transposes)."""
    lib = _lib.load()
    srcs = list(srcs) if isinstance(srcs, (list, tuple)) else [srcs]
    _require_cuda(g, "g")
    op = g.dtype
    if op not in _OPS16 or any(t.dtype != op for t in srcs) or not 1 <= len(srcs) <= 4:
        raise _lib.GmlmError("gemm_tn: one to four sources, all operands bfloat16 or all float16")
    m, n = int(g.size(0)), int(g.size(1))
    if any(t.dim() != 2 or t.size(0) != m for t in srcs):
        raise _lib.GmlmError("gemm_tn: row count mismatch")
    srcs = [_tma_rows(t) for t in srcs]
    g = _tma_rows(g)
    dev = g.device
    k = len(srcs)
    ka = sum(int(t.size(1)) for t in srcs)
    with torch.cuda.device(dev):
        out = torch.empty((ka, _rup(n, 4)), dtype=torch.float32, device=dev)
        ptrs = (C.c_void_p * k)(*[t.data_ptr() for t in srcs])
        ldas = (C.c_int64 * k)(*[_ld(t) for t in srcs])
        ks = (C.c_int64 * k)(*[int(t.size(1)) for t in srcs])
        ws_bytes = lib.gmlm_gemm_tn_workspace_bytes(k, ks, m, n)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.check(lib.gmlm_gemm_tn(k, ptrs, ldas, ks, _ptr(g), _ld(g), m, n, _ptr(out), out.size(1), _op_code(op),
                                    _ptr(ws), ws_bytes, _stream(dev)), "gemm_tn")
    return out if out.size(1) == n else out[:, :n]


# ------------------------------------------------------------------------------ A4 basis composition
def _rup(v: int, q: int) -> int:
    return (v + q - 1) // q * q


def basis_compose(weight: torch.Tensor, comp: Optional[torch.Tensor], root: Optional[torch.Tensor], live: Sequence[int],
                  op_dtype: torch.dtype, layout: str = "agg", want_n: bool = True, want_t: bool = True):
    """A4 in one pass over the fp32 bases: the composed weights of the populated relations ``live`` (+ ``root`` as one
    more slab), written in ``op_dtype`` in the two layouts the dense transforms consume.

    layout "agg" (aggregate-first layer, K = (S+1)*Fi):  wn [K, Fo] = [W_0; ..; W_{S-1}; root],  wt [Fo, K] = wn^T
    layout "tf"  (transform-first layer):                wn [Fi, (S+1)*Fo] = [W_0 | .. | root],  wt = wn^T
    Both are views with a 16-byte row pitch.  No autograd (see ``basis_compose_bwd``)."""
    lib = _lib.load()
    _require_cuda(weight, "weight")
    nb, fi, fo = (int(v) for v in weight.shape)
    S = len(live)
    slabs = S + (1 if root is not None else 0)
    per = 16 // torch.empty((), dtype=op_dtype).element_size()
    dev = weight.device
    w32 = weight.detach().float().contiguous()
    c32 = comp.detach().float().contiguous() if comp is not None else None
    r32 = root.detach().float().contiguous() if root is not None else None
    rels = (C.c_int32 * max(S, 1))(*[int(v) for v in live])
    with torch.cuda.device(dev):
        if layout == "agg":
            k = slabs * fi
            ldn, ldt = _rup(fo, per), _rup(k, per)
            wn = torch.empty((k, ldn), dtype=op_dtype, device=dev)[:, :fo] if want_n else None
            wt = torch.empty((fo, ldt), dtype=op_dtype, device=dev)[:, :k] if want_t else None
            n_args = (fi * ldn, ldn, S * fi * ldn)
            t_args = (fi, ldt, S * fi)
        elif layout == "tf":
            k = slabs * fo
            ldn, ldt = _rup(k, per), _rup(fi, per)
            wn = torch.empty((fi, ldn), dtype=op_dtype, device=dev)[:, :k] if want_n else None
            wt = torch.empty((k, ldt), dtype=op_dtype, device=dev)[:, :fi] if want_t else None
            n_args = (fo, ldn, S * fo)
            t_args = (fo * ldt, ldt, S * fo * ldt)
        else:
            raise _lib.GmlmError(f"basis_compose: unknown layout {layout!r}")
        _lib.check(lib.gmlm_basis_compose(_ptr(c32), _ptr(w32), _ptr(r32), rels, S,
                                          int(comp.size(0)) if comp is not None else nb, nb, fi, fo, _op_code(op_dtype),
                                          _ptr(wn), *n_args, _ptr(wt), *t_args, _stream(dev)), "basis_compose")
    return wn, wt


def basis_compose_bwd(weight: torch.Tensor, comp: Optional[torch.Tensor], dw: torch.Tensor, slot_stride: int,
                      row_stride: int, live: Sequence[int], need_weight: bool = True, need_comp: bool = True):
    """Gradients of the composition: ``dw`` = fp32 gradient of the composed weights of the populated relations in
    the natural strided layout ``dw[s*slot_stride + i*row_stride + o]``.  Returns (dweight [B,Fi,Fo], dcomp [R,B]).
    Shapes the kernel does not take (more than 8 populated relations, Fo or a stride not a multiple of 4) run as two
    stock torch matmuls."""
    lib = _lib.load()
    nb, fi, fo = (int(v) for v in weight.shape)
    S = len(live)
    dev = weight.device
    if comp is None:                       # no basis decomposition: the gradient slabs ARE the weight gradient
        dweight = torch.zeros_like(weight, dtype=torch.float32)
        flat = dw.reshape(-1)
        for s, r in enumerate(live):
            dweight[r] = torch.as_strided(flat, (fi, fo), (row_stride, 1), s * slot_stride)
        return dweight, None
    if S and not (S <= 8 and fo % 4 == 0 and slot_stride % 4 == 0 and row_stride % 4 == 0):
        dws = torch.as_strided(dw, (S, fi, fo), (slot_stride, row_stride, 1)).reshape(S, fi * fo)
        dweight = (comp.detach().float()[list(live)].t() @ dws).view_as(weight) if need_weight else None
        dcomp = None
        if need_comp:
            dcomp = torch.zeros_like(comp, dtype=torch.float32)
            dcomp[list(live)] = dws @ weight.detach().float().view(nb, -1).t()
        return dweight, dcomp
    w32 = weight.detach().float().contiguous()
    c32 = comp.detach().float().contiguous()
    R = int(comp.size(0))
    rels = (C.c_int32 * max(S, 1))(*[int(v) for v in live])
    with torch.cuda.device(dev):
        dweight = torch.empty((nb, fi, fo), dtype=torch.float32, device=dev) if need_weight else None
        dcomp = torch.empty((R, nb), dtype=torch.float32, device=dev) if need_comp else None
        if S == 0:
            return (dweight.zero_() if need_weight else None), (dcomp.zero_() if need_comp else None)
        ws_bytes = lib.gmlm_basis_compose_bwd_workspace_bytes(S, R, nb, fi, fo)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.check(lib.gmlm_basis_compose_bwd(_ptr(c32), _ptr(w32), _ptr(dw), int(slot_stride), int(row_stride), rels,
                                              S, R, nb, fi, fo, _ptr(dweight), _ptr(dcomp), _ptr(ws), ws_bytes,
                                              _stream(dev)), "basis_compose_bwd")
    return dweight, dcomp


def _to(t: Optional[torch.Tensor], dtype: Optional[torch.dtype]) -> Optional[torch.Tensor]:
    return t.to(dtype) if t is not None else None


def _gemm_nt_runs(op: torch.dtype, out_dtype: torch.dtype, cuda: bool, stock: bool) -> bool:
    """Whether a dense product of the RGCN layers runs on ``gemm_nt`` (tcgen05 for 16-bit operands, 3xTF32 for fp32
    ones) rather than on stock cuBLAS.  ``gemm_nt`` cannot write bf16 from fp32 operands, so with fp32 activations and
    a bf16 layer output the forward runs on cuBLAS while the backward's dh / dx, fp32 like the activations, run on
    3xTF32.  ``stock`` (``RGCNConv.use_tcgen05 = False``, fp32 operands) keeps every product on cuBLAS."""
    return op in _OPS16 or (op == torch.float32 and cuda and out_dtype == torch.float32 and not stock)


def _dense_nt(srcs, b: torch.Tensor, out_dtype: torch.dtype, on_gemm_nt: bool, bias=None, split: int = 0):
    """``[srcs] @ b.T (+ bias)`` in ``out_dtype`` on the engine ``_gemm_nt_runs`` chose; ``split`` > 0 returns the
    output's columns before and after ``split`` as two tensors.  On cuBLAS every source is its own matmul over its
    columns of ``b``, accumulated into the first in fp32."""
    if on_gemm_nt:
        return gemm_nt(srcs, b, bias=bias, out_dtype=out_dtype, split=split)
    a = srcs[0]
    if split:
        return (a @ b[:split].t()).to(out_dtype), (a @ b[split:].t()).to(out_dtype)
    k = a.size(1)
    out = a @ b[:, :k].t() if bias is None else torch.addmm(bias.float(), a, b[:, :k].t())
    for s in srcs[1:]:
        out.addmm_(s, b[:, k:k + s.size(1)].t())
        k += s.size(1)
    return out.to(out_dtype)


def _mm_f32(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """a @ b with an fp32 result for a parameter gradient (a reduction over up to millions of rows must not be
    rounded to 8 mantissa bits before it reaches the fp32 parameter)."""
    if a.dtype == torch.float32:
        return a @ b
    try:
        return torch.mm(a, b, out_dtype=torch.float32)
    except (TypeError, RuntimeError):
        return (a @ b).float()


_ONES: dict = {}


def _ones_source(m: int, dtype: torch.dtype, dev: torch.device) -> torch.Tensor:
    """[M, 8] of ones: appended as one more source of a weight-gradient reduction, its rows of the result are the
    column sums of g = the bias gradient, so the reduction that already streams g produces it (no extra pass)."""
    key = (m, dtype, dev)
    t = _ONES.get(key)
    if t is None:
        if len(_ONES) > 8:
            _ONES.clear()
        t = _ONES[key] = torch.ones((m, 8), dtype=dtype, device=dev)
    return t


def _param_grads(srcs, g: torch.Tensor, need, bias: bool, bias_col: int = 0):
    """fp32 parameter gradients of a product ``[srcs] @ W + bias`` with output gradient ``g``: ``[s^T g for s in srcs]``
    (None for a source not computed) and the bias gradient ``1^T g[:, bias_col:]`` (None unless ``bias``).

    16-bit operands: when any of ``need`` is set, ONE tcgen05 reduction over every source, with the ones source for the
    bias when at most three sources leave room for it.  fp32 operands: ``_mm_f32`` for each source ``need`` marks.  A
    bias gradient the reduction did not produce is a column sum: one pass, fp64 accumulation, fixed order."""
    grads, dbias = [None] * len(srcs), None
    if g.dtype in _OPS16:
        if any(need):
            with_ones = bias and len(srcs) < 4
            d = gemm_tn(list(srcs) + ([_ones_source(g.size(0), g.dtype, g.device)] if with_ones else []), g)
            k = 0
            for i, s in enumerate(srcs):
                grads[i] = d[k:k + s.size(1)]
                k += s.size(1)
            if with_ones:
                dbias = d[k, bias_col:]
    else:
        grads = [_mm_f32(s.t(), g) if n else None for s, n in zip(srcs, need)]
    if bias and dbias is None:
        gc = g[:, bias_col:]
        dbias = torch.ops.gmlm.colstats(gc if gc.dtype in _DT else gc.float())[0]
    return grads, dbias


class _RGCNTransform(torch.autograd.Function):
    """out = [h | x] @ [W_live ; root] + bias  (A4 + A6) for an aggregate-first layer.

    The composed weights never exist as a torch tensor: ``basis_compose`` reads the fp32 bases once and writes the
    GEMM's B operand in both layouts; 16-bit operand types run ONE tcgen05 GEMM over the two A sources (bias in the
    epilogue); fp32 operands run as 3xTF32 or on cuBLAS (``_gemm_nt_runs``).  Backward: [dh | dx] = g @ [W;root]^T
    is one more launch of the same kernel with two output maps (dh lands contiguous for the transposed aggregation);
    dW = h^T g and droot = x^T g are reductions over all nodes, produced in fp32; ``basis_compose_bwd`` turns dW
    into the basis and coefficient gradients in one pass over the bases.

    ``op_dtype``: bf16 for the bf16 pipeline, fp16 under ``torch.amp.autocast`` (what the reference's matmuls run in,
    main.py:446,543); h and x are cast once and saved in that type."""

    @staticmethod
    def forward(ctx, h, x, weight, comp, root, bias, live, out_dtype, op_dtype, stock=False):
        live = tuple(int(v) for v in live)
        S, fi, fo = len(live), weight.size(1), weight.size(2)
        k1 = S * fi
        ctx.stock = bool(stock)       # fp32 on stock cuBLAS (A/B switch RGCNConv.use_tcgen05 = False)
        # fp32 activations outside autocast (the reference's eval mode, main.py:603) run the same ONE GEMM with fp32
        # operands on the tf32 tensor cores as 3xTF32 (fp32-grade accuracy) when the output is fp32
        nt = _gemm_nt_runs(op_dtype, out_dtype, h.is_cuda, stock)
        srcs = [h] + ([x] if root is not None else [])
        srcs = [_tma_rows(t, op_dtype) if nt else t.float() for t in srcs]
        wn, wt = basis_compose(weight, comp, root, live, op_dtype, "agg",
                               want_n=any(ctx.needs_input_grad[:2]) or not nt, want_t=nt)
        out = _dense_nt(srcs, wt if nt else wn.t(), out_dtype, nt, bias=bias)
        hq, xq = srcs[0], (srcs[1] if root is not None else None)
        ctx.save_for_backward(hq, xq, wn, weight, comp)
        ctx.live, ctx.k1, ctx.op = live, k1, op_dtype
        ctx.dtypes = (weight.dtype, None if comp is None else comp.dtype, None if root is None else root.dtype,
                      None if bias is None else bias.dtype, h.dtype, x.dtype)
        return out

    @staticmethod
    def backward(ctx, g):
        hq, xq, wn, weight, comp = ctx.saved_tensors
        k1, live, op, needs = ctx.k1, ctx.live, ctx.op, ctx.needs_input_grad
        fi, fo = weight.size(1), weight.size(2)
        need_h, need_x = needs[0], needs[1] and xq is not None
        dh = dx = dweight = dcomp = None
        gb = g if (g.dtype == op and g.is_contiguous()) else g.to(op).contiguous()
        if need_h or need_x:
            out_dt = torch.bfloat16 if op in _OPS16 and ctx.dtypes[4] == torch.bfloat16 else torch.float32
            nt = _gemm_nt_runs(op, out_dt, gb.is_cuda, ctx.stock)
            if need_h and need_x:
                dh, dx = _dense_nt([gb], wn, out_dt, nt, split=k1)             # [M, Fo] x [K1+K2, Fo]^T
            elif need_h:
                dh = _dense_nt([gb], wn[:k1], out_dt, nt)
            else:
                dx = _dense_nt([gb], wn[k1:], out_dt, nt)
            dh = _to(dh.contiguous(), ctx.dtypes[4]) if dh is not None else None
            dx = _to(dx, ctx.dtypes[5])
        # dW = h^T g [S*Fi, Fo], droot = x^T g and dbias = 1^T g, fp32
        need_w = needs[2] or needs[3]
        (dw, *dr), dbias = _param_grads([hq] + ([xq] if xq is not None else []), gb, [need_w, needs[4]], needs[5])
        if need_w:
            dweight, dcomp = basis_compose_bwd(weight, comp, dw.contiguous(), fi * fo, fo, live, needs[2],
                                               needs[3] and comp is not None)
        droot = _to(dr[0].contiguous(), ctx.dtypes[2]) if needs[4] and xq is not None else None
        return (dh, dx, _to(dweight, ctx.dtypes[0]), _to(dcomp, ctx.dtypes[1]), droot, _to(dbias, ctx.dtypes[3]),
                None, None, None, None)


class _RGCNSegCompact(torch.autograd.Function):
    """RGCNConv on the SEGMENT-COMPACT view of the graph (``RelGraph.seg_plan``; A5 + A4 + A6 of one layer):

        H_c   = mean over the edges of every NON-EMPTY (dst, slot) segment            [rows_c, Fi]   (slot-major)
        out   = x @ root + bias;   out[dst of slot s's rows] += H_c[slot s] @ W_s      one GEMM per populated slot

    The dense form multiplies the zero rows of H: on the reference's own graphs most (dst, rel) segments are empty
    (Roman-empire shape: 22.7k nodes x 4 slots = 90.6k segments, at most 32.9k with an edge), and at the shipped widths
    (H = 512) the layer is FLOP-bound, so half of the forward, the [dH | dx] and the dW products are spent on zeros.
    Here every product runs over the compact rows only.  Backward: g rows gathered per slot, dH_c = g_s @ W_s^T,
    dW_s = H_c[s]^T g_s, [droot; dbias] = [x | 1]^T g, dx = g @ root^T + (transposed compact aggregation of dH_c).
    A compact row's edges keep their CSR order, so H_c equals the dense H's rows bit for bit; the per-destination sum
    over slots runs in slot order (the dense GEMM sums along K in the same slot order, with other roundings)."""

    @staticmethod
    def forward(ctx, x, weight, comp, root, bias, plan, num_nodes, live, out_dtype, op_dtype):
        live = tuple(int(v) for v in live)
        S, fi, fo = len(live), weight.size(1), weight.size(2)
        h_c = _spmm_csr(x, plan.fwd, _lib.AGG_MEAN)
        hq = _tma_rows(h_c, op_dtype)
        xq = _tma_rows(x[:num_nodes], op_dtype)
        wn, wt = basis_compose(weight, comp, root, live, op_dtype, "agg")
        out = gemm_nt(xq, wt[:, S * fi:], bias=bias, out_dtype=out_dtype)          # root term + bias
        for s in range(S):
            a, c = plan.slot_start[s], plan.slot_count[s]
            if c:
                y = gemm_nt(hq[a:a + c], wt[:, s * fi:(s + 1) * fi], out_dtype=out_dtype)
                scatter_add_rows_(out, plan.dst[a:a + c], y)
        ctx.save_for_backward(hq, xq, wn, weight, comp)
        ctx.plan, ctx.live, ctx.op, ctx.num_nodes = plan, live, op_dtype, num_nodes
        ctx.dtypes = (weight.dtype, None if comp is None else comp.dtype, root.dtype,
                      None if bias is None else bias.dtype, x.dtype)
        ctx.num_src = x.size(0)
        return out

    @staticmethod
    def backward(ctx, g):
        hq, xq, wn, weight, comp = ctx.saved_tensors
        plan, live, op, n = ctx.plan, ctx.live, ctx.op, ctx.num_nodes
        S, fi, fo = len(live), weight.size(1), weight.size(2)
        g = g.contiguous()
        gq = _tma_rows(g, op)
        acc_dt = torch.bfloat16 if ctx.dtypes[4] == torch.bfloat16 else torch.float32
        dx = dweight = dcomp = None
        need_x = ctx.needs_input_grad[0]
        need_w = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        g_src = g if g.dtype in _DT else g.float()                         # the row gather takes fp32 / bf16
        dh_parts, dw = [], None
        if need_w:
            dw = torch.zeros((S * fi, fo), dtype=torch.float32, device=g.device)
        rows_done = 0
        for s in range(S):
            a, c = plan.slot_start[s], plan.slot_count[s]
            pad = (plan.slot_start[s + 1] if s + 1 < S else plan.num_rows) - a - c
            if c:
                gs = _tma_rows(gather_rows(g_src, plan.dst[a:a + c]), op)
                if need_x:
                    dh_parts.append(gemm_nt(gs, wn[s * fi:(s + 1) * fi], out_dtype=acc_dt))
                if need_w:
                    dw[s * fi:(s + 1) * fi] = gemm_tn([hq[a:a + c]], gs)
            if need_x and pad:
                dh_parts.append(torch.zeros((pad, fi), dtype=acc_dt, device=g.device))
            rows_done = a + c + pad
        if need_x:
            dh_c = torch.cat(dh_parts, dim=0) if dh_parts else torch.zeros((0, fi), dtype=acc_dt, device=g.device)
            if dh_c.size(0) == 0:                                                         # a graph without edges
                dx = torch.zeros((ctx.num_src, fi), dtype=acc_dt, device=g.device)
            else:
                dx = _spmm_csr(dh_c, plan.bwd, _lib.AGG_WEIGHTED)                         # [num_src, Fi]
            dxr = gemm_nt(gq, wn[S * fi:], out_dtype=acc_dt)                              # root term, local rows
            if dx.size(0) == dxr.size(0):
                dx = dx + dxr
            else:
                dx[:n] += dxr
            dx = dx.to(ctx.dtypes[4])
        # [droot; dbias] = [x | 1]^T g in one reduction, also when only the bias needs it
        (droot,), dbias = _param_grads([xq], gq, [ctx.needs_input_grad[3] or ctx.needs_input_grad[4]],
                                       ctx.needs_input_grad[4])
        droot = _to(droot.contiguous(), ctx.dtypes[2]) if ctx.needs_input_grad[3] else None
        if need_w:
            dweight, dcomp = basis_compose_bwd(weight, comp, dw, fi * fo, fo, live, ctx.needs_input_grad[1],
                                               ctx.needs_input_grad[2] and comp is not None)
        return (dx, _to(dweight, ctx.dtypes[0]), _to(dcomp, ctx.dtypes[1]), droot, _to(dbias, ctx.dtypes[3]),
                None, None, None, None, None)


def rgcn_segment_compact(x: torch.Tensor, graph: RelGraph, weight: torch.Tensor, comp: Optional[torch.Tensor],
                         root: torch.Tensor, bias: Optional[torch.Tensor],
                         out_dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """RGCNConv over the non-empty segments only (see ``_RGCNSegCompact``); 16-bit operand types."""
    _require_cuda(x, "x")
    op, out_dt = _dense_dtypes(x, out_dtype)
    if op not in _OPS16 or out_dt not in _DT:
        raise _lib.GmlmError("rgcn_segment_compact: 16-bit operand types (bf16 pipeline or autocast) only")
    if x.dtype not in _DT:
        x = x.float()
    with torch.amp.autocast("cuda", enabled=False):
        return _RGCNSegCompact.apply(x, weight, comp, root, bias, graph.seg_plan(), graph.num_nodes,
                                     tuple(graph.live_rels), out_dt, op)


class _RGCNTransformFirst(torch.autograd.Function):
    """Z = x @ [W_0 | .. | W_{S-1} | root] (+ bias on the root slab) for a transform-first layer (A4 + A6): the same
    composition kernel in the "tf" layout, the same GEMM; backward dx = dZ @ [W | root]^T, dW = x^T dZ (fp32)."""

    @staticmethod
    def forward(ctx, x, weight, comp, root, bias, live, out_dtype, op_dtype, stock=False):
        live = tuple(int(v) for v in live)
        S, fi, fo = len(live), weight.size(1), weight.size(2)
        bias_cat = None
        if bias is not None:
            bias_cat = torch.cat([bias.new_zeros(S * fo), bias.detach()]).float()
        ctx.stock = bool(stock)
        nt = _gemm_nt_runs(op_dtype, out_dtype, x.is_cuda, stock)
        xq = _tma_rows(x, op_dtype) if nt else x.float()
        wn, wt = basis_compose(weight, comp, root, live, op_dtype, "tf", want_n=ctx.needs_input_grad[0] or not nt,
                               want_t=nt)
        z = _dense_nt([xq], wt if nt else wn.t(), out_dtype, nt, bias=bias_cat)
        ctx.save_for_backward(xq, wn, weight, comp)
        ctx.live, ctx.op = live, op_dtype
        ctx.dtypes = (weight.dtype, None if comp is None else comp.dtype, root.dtype,
                      None if bias is None else bias.dtype, x.dtype)
        return z

    @staticmethod
    def backward(ctx, gz):
        xq, wn, weight, comp = ctx.saved_tensors
        live, op, needs = ctx.live, ctx.op, ctx.needs_input_grad
        S, fo = len(live), weight.size(2)
        dx = dweight = dcomp = droot = None
        gb = gz if (gz.dtype == op and gz.is_contiguous()) else gz.to(op).contiguous()
        if needs[0]:
            out_dt = torch.bfloat16 if op in _OPS16 and ctx.dtypes[4] == torch.bfloat16 else torch.float32
            dx = _to(_dense_nt([gb], wn, out_dt, _gemm_nt_runs(op, out_dt, gb.is_cuda, ctx.stock)).contiguous(),
                     ctx.dtypes[4])
        # dWn = x^T dZ [Fi, (S+1)*Fo] fp32; the bias is on the root slab only
        (dwn,), dbias = _param_grads([xq], gb, [any(needs[1:4])], needs[4], bias_col=S * fo)
        if needs[1] or needs[2]:
            dwn = dwn.contiguous()
            dweight, dcomp = basis_compose_bwd(weight, comp, dwn, fo, dwn.size(1), live, needs[1],
                                               needs[2] and comp is not None)
        if needs[3]:
            droot = _to(dwn[:, S * fo:].contiguous(), ctx.dtypes[2])
        return (dx, _to(dweight, ctx.dtypes[0]), _to(dcomp, ctx.dtypes[1]), droot, _to(dbias, ctx.dtypes[3]),
                None, None, None, None)


class _LinearNT(torch.autograd.Function):
    """y = [x_0 | x_1 | ..] @ wt.T + bias (+ addend) on the tcgen05 GEMM (16-bit operands, fp32 accumulation).  The
    sources are never concatenated (MultiScaleFusion, main.py:176-180); ``addend`` is a residual folded into the
    epilogue (main.py:281-282).  Backward: dx on the same kernel, weight gradient as an fp32 reduction."""

    @staticmethod
    def forward(ctx, wt, bias, addend, out_dtype, op_dtype, *xs):
        xq = [_tma_rows(x, op_dtype) for x in xs]
        wtq = _tma_rows(wt.detach(), op_dtype)                            # [N_out, K]
        if addend is not None and addend.dtype != out_dtype:
            addend = addend.to(out_dtype)
        y = gemm_nt(xq, wtq, bias=bias, out_dtype=out_dtype, addend=addend)
        ctx.save_for_backward(wtq, *xq)
        ctx.dtypes = (wt.dtype, None if bias is None else bias.dtype, [x.dtype for x in xs])
        ctx.op = op_dtype
        return y

    @staticmethod
    def backward(ctx, g):
        wtq, *xq = ctx.saved_tensors
        op = ctx.op
        gb = g if (g.dtype == op and g.is_contiguous()) else g.to(op).contiguous()
        dwt = dadd = None
        dxs = [None] * len(xq)
        if any(ctx.needs_input_grad[5:]):
            all_bf16 = all(d == torch.bfloat16 for d in ctx.dtypes[2])
            widths = [int(x.size(1)) for x in xq]
            odt = torch.bfloat16 if all_bf16 else torch.float32
            wt_t = wtq.t().contiguous()
            if len(widths) <= 2 or all(v % 64 == 0 for v in widths[:-1]):
                # one launch, one CONTIGUOUS gradient per source (epilogue chunks routed to up to four tensor maps):
                # autograd's sums with the other gradients of a layer output stay vectorised
                parts = gemm_nt(_tma_rows(gb), wt_t, out_dtype=odt, split=widths)
            else:
                dx = gemm_nt(_tma_rows(gb), wt_t, out_dtype=odt)
                parts, k0 = [], 0
                for v in widths:
                    parts.append(dx[:, k0:k0 + v])
                    k0 += v
            for i, d in enumerate(parts):
                if ctx.needs_input_grad[5 + i]:
                    dxs[i] = d.to(ctx.dtypes[2][i])
        # dWt = g^T [x_0 | x_1 | ..] as ([x..]^T g)^T: one tcgen05 reduction over the sources (+ 1^T g = dbias)
        dws, dbias = _param_grads(xq, gb, [ctx.needs_input_grad[0]] * len(xq), ctx.needs_input_grad[1])
        if ctx.needs_input_grad[0]:
            dwt = torch.cat([d.t() for d in dws], dim=1).to(ctx.dtypes[0])
        if ctx.needs_input_grad[2]:
            dadd = g
        return (dwt, _to(dbias, ctx.dtypes[1]), dadd, None, None, *dxs)


def linear_nt(x, wt: torch.Tensor, bias: Optional[torch.Tensor] = None, out_dtype: Optional[torch.dtype] = None,
              op_dtype: Optional[torch.dtype] = None, addend: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``F.linear(cat(x, 1), wt, bias) + addend`` on the tcgen05 GEMM; ``x`` one tensor or a list of up to four
    sources.  ``op_dtype``: operand type (default: x's when 16-bit, else bf16); ``out_dtype``: bf16 or fp32."""
    xs = list(x) if isinstance(x, (list, tuple)) else [x]
    op = op_dtype or (xs[0].dtype if xs[0].dtype in _OPS16 else torch.bfloat16)
    out_dtype = out_dtype or (torch.bfloat16 if xs[0].dtype == torch.bfloat16 else torch.float32)
    return _LinearNT.apply(wt, bias, addend, out_dtype, op, *xs)


def _dense_dtypes(x: torch.Tensor, out_dtype: Optional[torch.dtype]):
    """(operand type, output type) of a dense transform called with activations x: the autocast type with fp32
    results under torch.amp.autocast (upstream accumulates into an fp32 `out`), bf16 in the bf16 pipeline, fp32
    otherwise."""
    if torch.is_autocast_enabled("cuda"):
        return torch.get_autocast_dtype("cuda"), out_dtype or torch.get_default_dtype()
    if x.dtype == torch.bfloat16:
        return torch.bfloat16, out_dtype or torch.get_default_dtype()
    return torch.float32, out_dtype or torch.get_default_dtype()


def rgcn_transform_first(x: torch.Tensor, graph: RelGraph, weight: torch.Tensor, comp: Optional[torch.Tensor],
                         root: torch.Tensor, bias: Optional[torch.Tensor], out_dtype: Optional[torch.dtype] = None,
                         use_tcgen05: bool = True) -> torch.Tensor:
    """RGCNConv as TRANSFORM-then-aggregate (A5+A6 fused by linearity of the mean; include/gmlm_b200.h
    ``gmlm_dst_plan``):  Z = x @ [W_0 | .. | W_{S-1} | root] (+ bias on the root slab),
    out[i] = sum_e w_e Z[src_e, slot_e] + Z[i, S].  The [N, S*Fi] matrix H of the aggregate-first form is never
    materialised and the gather moves Fo-wide rows instead of Fi-wide ones.

    x [num_src, Fi]; weight [B, Fi, Fo] / comp [R, B] (the layer's parameters); root [Fi, Fo]."""
    _require_cuda(x, "x")
    live = graph.live_rels
    S, fi, fo = len(live), int(weight.size(1)), int(weight.size(2))
    if S != graph.num_slots or x.size(0) != graph.num_src or x.size(1) != fi:
        raise _lib.GmlmError("rgcn_transform_first: shape mismatch")
    fplan, bplan = graph.dst_plan()
    op, out_dt = _dense_dtypes(x, out_dtype)
    if not use_tcgen05:
        op = torch.float32
    z_dt = out_dt if out_dt in _DT else torch.float32          # the gather kernels take fp32 / bf16
    with torch.amp.autocast("cuda", enabled=False):
        z = _RGCNTransformFirst.apply(x, weight, comp, root, bias, tuple(live), z_dt, op, not use_tcgen05)
        fl, fm = csr_pack(fplan)
        bl, bm = csr_pack(bplan)
        # one Fo-wide row per (node, slab); a GEMM output whose row pitch is padded to 16 bytes is copied first
        out = torch.ops.gmlm.plan_aggregate(z.reshape(graph.num_src * (S + 1), fo), *fl, *bl, fm + bm)
    return out if out.dtype == out_dt else out.to(out_dt)


def rgcn_transform(h: torch.Tensor, x: torch.Tensor, weight: torch.Tensor, comp: Optional[torch.Tensor],
                   root: Optional[torch.Tensor], bias: Optional[torch.Tensor], live: Sequence[int],
                   out_dtype: Optional[torch.dtype] = None, use_tcgen05: bool = True) -> torch.Tensor:
    """A4 + A6 of an aggregate-first layer: ``[h | x] @ [W_live ; root] + bias`` (see ``_RGCNTransform``)."""
    op, out_dt = _dense_dtypes(h, out_dtype)
    if not use_tcgen05:
        op = torch.float32
    with torch.amp.autocast("cuda", enabled=False):
        return _RGCNTransform.apply(h, x, weight, comp, root, bias, tuple(live), out_dt, op, not use_tcgen05)


# ------------------------------------------------------------------------------ halo pack / unpack
def gather_rows(x: torch.Tensor, ids: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[k] = x[ids[k]] (pack the rows a peer needs)."""
    lib = _lib.load()
    _require_cuda(x, "x")
    x = _rowmajor(x)
    ids = ids.contiguous()
    n, feat = int(ids.numel()), int(x.size(1))
    with torch.cuda.device(x.device):
        if out is None:
            out = torch.empty((n, feat), dtype=x.dtype, device=x.device)
        _lib.check(lib.gmlm_gather_rows(_ptr(x), _dtype_code(x, "gather_rows"), feat, _ld(x), _ptr(ids), n, _ptr(out),
                                        _ld(out) if n > 1 else feat, _stream(x.device)), "gather_rows")
    return out


def scatter_add_rows_(dst: torch.Tensor, ids: torch.Tensor, src: torch.Tensor) -> torch.Tensor:
    """dst[ids[k]] += src[k] in place; ``ids`` must be unique (no atomics, deterministic)."""
    lib = _lib.load()
    _require_cuda(dst, "dst")
    if dst.dim() != 2 or dst.stride(1) != 1 or src.dim() != 2 or src.stride(1) != 1:
        raise _lib.GmlmError("scatter_add_rows_: row-major 2-D tensors required")
    ids = ids.contiguous()
    n, feat = int(ids.numel()), int(dst.size(1))
    with torch.cuda.device(dst.device):
        _lib.check(lib.gmlm_scatter_add_rows(_ptr(dst), _dtype_code(dst, "scatter_add_rows"), feat, _ld(dst), _ptr(ids),
                                             n, _ptr(src), _ld(src) if n > 1 else feat, _stream(dst.device)),
                   "scatter_add_rows")
    return dst


# ------------------------------------------------------------------------------ public functional API
def degree(index: torch.Tensor, num_nodes: Optional[int] = None, dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """Drop-in for ``torch_geometric.utils.degree`` (``/root/reference/main.py:7``; called
    ``main.py:65,256``): float32 [N] occurrence counts of ``index``."""
    _require_cuda(index, "index")
    if num_nodes is None:  # upstream maybe_num_nodes (one host sync)
        num_nodes = int(index.max()) + 1 if index.numel() > 0 else 0
    deg = torch.ops.gmlm.degree_i32(index, int(num_nodes))
    return deg.to(dtype or torch.get_default_dtype())


def edge_type_from_degree(edge_index: torch.Tensor, num_nodes: int, bounds: Sequence[int] = (2, 5, 10)) -> torch.Tensor:
    """The reference's per-edge loop ``main.py:253-267`` as one kernel: relation id =
    bucket of the source node's out-degree (<=2, <=5, <=10, else)."""
    _require_cuda(edge_index, "edge_index")
    src = edge_index[0]
    deg = torch.ops.gmlm.degree_i32(src, int(num_nodes))
    return torch.ops.gmlm.edge_type_bucket(src, deg, list(bounds))


def rgcn_aggregate(x: torch.Tensor, graph: RelGraph) -> torch.Tensor:
    """Per-(dst, relation) mean of source rows: ``[N, F] -> [N, S*F]`` (S = populated relations).
    Forward = A5, backward = A14 (gather on the transposed CSR with 1/count folded in)."""
    _require_cuda(x, "x")
    if x.size(0) != graph.num_src:
        raise _lib.GmlmError(f"x has {x.size(0)} rows, graph has {graph.num_src} source nodes")
    fl, fm = csr_pack(graph.fwd)
    bl, bm = csr_pack(graph.bwd)
    return torch.ops.gmlm.rgcn_aggregate(x, *fl, *bl, fm + bm + [int(graph.num_nodes), int(graph.num_slots)])


def graph_norm(x, weight, bias, mean_scale, eps: float = 1e-5, fuse_gelu: bool = False) -> torch.Tensor:
    _require_cuda(x, "x")
    return torch.ops.gmlm.graphnorm_fwd(x, weight, bias, mean_scale, float(eps), bool(fuse_gelu))[0]


def layer_norm(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    """``nn.LayerNorm(C)`` over the last dimension of a 2-D CUDA tensor (the ``self.layer_norm(fused)`` of
    ``MultiScaleFusion``, ``/root/reference/main.py:171,180``): one read + one write forward, two reads +
    one write backward, deterministic parameter gradients."""
    _require_cuda(x, "x")
    if not layer_norm_ok(x):
        raise _lib.GmlmError(f"layer_norm: unsupported input {tuple(x.shape)} {x.dtype} (see layer_norm_ok)")
    return torch.ops.gmlm.layernorm_fwd(x, weight, bias, float(eps))[0]


def soft_masking_gnn_input(x: torch.Tensor, gnn_perturb_mask: torch.Tensor, mask_token_embed: torch.Tensor,
                           beta: float = 0.7) -> torch.Tensor:
    """Drop-in for ``soft_masking_gnn_input`` (``/root/reference/main.py:92-99``): one fused pass,
    no clone + boolean-index round trip and no ``.any()`` host sync."""
    _require_cuda(x, "x")
    return torch.ops.gmlm.soft_mask_fwd(x, gnn_perturb_mask, mask_token_embed, float(beta))
