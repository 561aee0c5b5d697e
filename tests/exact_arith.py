"""Exact-arithmetic references for the aggregation, GEMM and basis-composition kernels.

Small integers as features and operands and powers of two as weights make every product exact, and every partial
sum exact in fp32 while it stays under 2^24 units of the smallest term.  The fp32 result is then the same for every
summation order, chunking, band order or split, so a kernel's output is fixed up to its last step -- the mean's
``acc * (1.0f / L)``, a GEMM epilogue's bias and addend, the store to bf16 / fp16 -- and that step is reproduced
here exactly.  Every ``expected_*`` function asserts its exactness budget before it returns, so a case outside the
budget fails in the reference, never in the comparison with the kernel.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np
import scipy.sparse as sp
import torch

AGG_SUM, AGG_MEAN, AGG_WEIGHTED = 0, 1, 2            # gmlm_b200._lib
FP32_EXACT = 1 << 24                                 # integers below this are exact in fp32
# tcgen05 kind::f16 / kind::tf32 products are exact; the accumulation aligns addends to the largest one and drops
# only bits below its ulp, so integer partial sums are kept below 2^22 units to leave that alignment two bits of room
TC_EXACT = 1 << 22
DYADIC = (-2.0, -1.0, -0.5, -0.25, 0.25, 0.5, 1.0, 2.0)


# ------------------------------------------------------------------------------ generators
def int_tensor(shape, dtype=torch.float32, lo: int = -4, hi: int = 4, nonzero: bool = False, seed: int = 0,
               device=None) -> torch.Tensor:
    """Integers in [lo, hi] (0 left out when ``nonzero``: a dropped term always shows), exact in ``dtype``."""
    rng = np.random.default_rng(seed)
    vals = np.arange(lo, hi + 1)
    if nonzero:
        vals = vals[vals != 0]
    assert max(abs(lo), abs(hi)) <= 256, "integers beyond 256 are not all exact in bf16"
    a = rng.choice(vals, size=shape).astype(np.float32)
    return torch.from_numpy(a).to(dtype=dtype, device=device)


def dyadic_weights(shape, seed: int = 0, device=None) -> torch.Tensor:
    """fp32 weights drawn from {+-1/4, +-1/2, +-1, +-2}."""
    rng = np.random.default_rng(seed)
    return torch.from_numpy(rng.choice(np.asarray(DYADIC, np.float32), size=shape)).to(device)


def pow2_graph(num_nodes: int, num_relations: int = 4, *, seed: int = 0, p_empty: float = 0.6, max_log: int = 3,
               hubs: Sequence[tuple] = (), fanout_sources: int = 0, fanout: int = 0):
    """(edge_index int64 [2, E], edge_type int64 [E]) whose non-empty (dst, rel) segments all have power-of-two
    lengths, so that the 1/|segment| weights of the backward and of the transform-first plan are dyadic.

    Ordinary segments: empty with probability ``p_empty``, else 2^k edges, k uniform in [0, max_log], sources
    uniform.  ``hubs``: (count, length) pairs: that many (dst, rel) segments get ``length`` (a power of two) edges
    with uniform sources -- on a large graph they gather from more rows than one band of the hub plan holds.
    ``fanout_sources`` sources each feed ``fanout`` distinct destinations through the last relation (one edge per
    segment, destinations disjoint between sources): rows of that length in the transposed CSR."""
    rng = np.random.default_rng(seed)
    r_ord = num_relations - 1 if fanout_sources else num_relations
    n_seg = num_nodes * r_ord
    lens = np.where(rng.random(n_seg) < p_empty, 0, 1 << rng.integers(0, max_log + 1, n_seg))
    taken = np.zeros(n_seg, bool)
    for count, length in hubs:
        assert length & (length - 1) == 0, "segment lengths must be powers of two"
        ids = rng.choice(np.nonzero(~taken)[0], size=count, replace=False)
        lens[ids] = length
        taken[ids] = True
    seg = np.repeat(np.arange(n_seg), lens)
    dst, rel = seg // r_ord, seg % r_ord
    src = rng.integers(0, num_nodes, seg.size)
    if fanout_sources:
        assert fanout_sources * fanout <= num_nodes
        d = rng.permutation(num_nodes)[:fanout_sources * fanout]
        s = np.repeat(rng.choice(num_nodes, fanout_sources, replace=False), fanout)
        src, dst = np.concatenate([src, s]), np.concatenate([dst, d])
        rel = np.concatenate([rel, np.full(d.size, num_relations - 1)])
    order = rng.permutation(src.size)                  # CSR order is not the generation order
    ei = torch.from_numpy(np.stack([src[order], dst[order]]).astype(np.int64))
    return ei, torch.from_numpy(rel[order].astype(np.int64))


# ------------------------------------------------------------------------------ budgets and rounding
def fraction_bits(a) -> int:
    """Fewest fraction bits q with every value of ``a`` a multiple of 2^-q (asserts that q <= 60 exists)."""
    v = np.abs(np.asarray(a, np.float64)).ravel()
    assert np.isfinite(v).all()
    for q in range(61):
        s = v * float(2 ** q)
        if np.all(s == np.floor(s)):
            return q
    raise AssertionError("values are not dyadic")


def check_budget(abs_sum, q: int, limit: int = FP32_EXACT, what: str = "") -> None:
    """Every partial sum of terms that are multiples of 2^-q, bounded by ``abs_sum``, is exact in the accumulator."""
    m = float(np.max(abs_sum)) if np.size(abs_sum) else 0.0
    assert m * 2.0 ** q < limit, f"{what}: sum |terms| = {m} in units of 2^-{q} leaves the exact range 2^{limit.bit_length() - 1}"


def round_to(a32: np.ndarray, dtype: torch.dtype) -> torch.Tensor:
    """fp32 -> ``dtype``, round to nearest, ties to even (the cvt.rn of the kernels' stores)."""
    a32 = np.ascontiguousarray(a32, np.float32)
    if dtype == torch.float32:
        return torch.from_numpy(a32.copy())
    if dtype == torch.float16:
        return torch.from_numpy(a32.astype(np.float16))
    assert dtype == torch.bfloat16
    assert np.isfinite(a32).all()
    u = a32.view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) >> 16
    return torch.from_numpy(u.astype(np.uint16).view(np.int16).copy()).view(torch.bfloat16)


def _np64(t: torch.Tensor) -> np.ndarray:
    return t.detach().double().cpu().numpy()


def _exact_f32(s: np.ndarray, what: str) -> np.ndarray:
    s32 = s.astype(np.float32)
    assert np.array_equal(s32.astype(np.float64), s), f"{what}: the exact value is not an fp32 number"
    return s32


# ------------------------------------------------------------------------------ aggregation
def expected_spmm(x: torch.Tensor, rowptr, col, mode: int, w: Optional[torch.Tensor] = None,
                  out_dtype: Optional[torch.dtype] = None, block_rows: int = 1 << 16) -> torch.Tensor:
    """What gmlm_spmm_csr writes: row r = sum over its edges of w[e] * x[col[e]] (w 1-D, or 2-D [nnz, H] with head
    h weighting features [h*F/H, (h+1)*F/H)), exact in fp64 and then in fp32; AGG_MEAN multiplies by
    fp32(1) / fp32(L) for rows of L > 1 edges; then one rounding into x's dtype.  CPU tensor."""
    out_dtype = out_dtype or x.dtype
    rp = np.asarray(rowptr.cpu() if torch.is_tensor(rowptr) else rowptr, np.int64)
    cl = np.asarray(col.cpu() if torch.is_tensor(col) else col, np.int64)
    xs = _np64(x)
    n_rows, feat = rp.size - 1, xs.shape[1]
    nnz = int(rp[-1])
    cl = cl[:nnz]
    q_x = fraction_bits(xs)
    if mode == AGG_WEIGHTED:
        wv = _np64(w)[:nnz]
        wv = wv[:, None] if wv.ndim == 1 else wv
    else:
        wv = np.ones((nnz, 1))
    heads = wv.shape[1]
    assert feat % heads == 0
    hw = feat // heads
    q = q_x + fraction_bits(wv)
    lens = np.diff(rp)
    outs = []
    for r0 in range(0, n_rows, block_rows):
        r1 = min(n_rows, r0 + block_rows)
        e0, e1 = rp[r0], rp[r1]
        s = np.empty((r1 - r0, feat))
        a = np.empty((r1 - r0, feat))
        for h in range(heads):
            m = sp.csr_matrix((wv[e0:e1, h], cl[e0:e1], rp[r0:r1 + 1] - e0), shape=(r1 - r0, xs.shape[0]))
            s[:, h * hw:(h + 1) * hw] = m @ xs[:, h * hw:(h + 1) * hw]
            m.data = np.abs(m.data)
            a[:, h * hw:(h + 1) * hw] = m @ np.abs(xs[:, h * hw:(h + 1) * hw])
        check_budget(a, q, what="spmm")
        s32 = _exact_f32(s, "spmm")
        if mode == AGG_MEAN:
            L = lens[r0:r1].astype(np.float32)
            scale = np.where(L > 1, np.float32(1) / np.maximum(L, np.float32(1)), np.float32(1)).astype(np.float32)
            s32 = s32 * scale[:, None]
        outs.append(round_to(s32, out_dtype))
    if not outs:
        return torch.zeros((0, feat), dtype=out_dtype)
    return torch.cat(outs)


def expected_csr_spmm(x: torch.Tensor, csr, mode: int) -> torch.Tensor:
    """``expected_spmm`` of a gmlm_b200 CSR (its own weights in weighted mode)."""
    return expected_spmm(x, csr.rowptr, csr.col, mode, csr.w if mode == AGG_WEIGHTED else None)


# ------------------------------------------------------------------------------ dense
def _epilogue(acc: np.ndarray, bias, addend, out_dtype, limit: int, abs_sum: np.ndarray, q: int, what: str):
    """fp32(acc) + bias, then + addend, each an fp32 add; one rounding into out_dtype."""
    check_budget(abs_sum, q, limit, what)
    v = _exact_f32(acc, what)
    if bias is not None:
        v = v + _np64(bias).astype(np.float32)[None, :]
    if addend is not None:
        v = v + _np64(addend).astype(np.float32)
    return round_to(v, out_dtype)


def expected_gemm(srcs, b: torch.Tensor, bias: Optional[torch.Tensor] = None, addend: Optional[torch.Tensor] = None,
                  out_dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """``gemm_nt``: [A_0 | A_1 | ..] @ b^T on the tensor cores (exact while the products stay under 2^22 units),
    then the fp32 epilogue: + bias, + addend, one rounding."""
    srcs = list(srcs) if isinstance(srcs, (list, tuple)) else [srcs]
    a = np.concatenate([_np64(t) for t in srcs], axis=1)
    bb = _np64(b)
    acc = a @ bb.T
    abs_sum = np.abs(a) @ np.abs(bb).T
    q = fraction_bits(a) + fraction_bits(bb)
    if bias is not None:
        check_budget(np.abs(acc) + np.abs(_np64(bias))[None, :], max(q, fraction_bits(_np64(bias))), FP32_EXACT,
                     "gemm bias")
    return _epilogue(acc, bias, addend, out_dtype, TC_EXACT, abs_sum, q, "gemm_nt")


def expected_gemm_tn(srcs, g: torch.Tensor) -> torch.Tensor:
    """``gemm_tn``: cat(srcs, 1)^T @ g, fp32, exact (every split partial and their sum stay under 2^22 units)."""
    srcs = list(srcs) if isinstance(srcs, (list, tuple)) else [srcs]
    a = np.concatenate([_np64(t) for t in srcs], axis=1)
    gg = _np64(g)
    acc = a.T @ gg
    abs_sum = np.abs(a).T @ np.abs(gg)
    return _epilogue(acc, None, None, torch.float32, TC_EXACT, abs_sum, fraction_bits(a) + fraction_bits(gg),
                     "gemm_tn")


def expected_compose(weight: torch.Tensor, comp: Optional[torch.Tensor], root: Optional[torch.Tensor],
                     live: Sequence[int], op_dtype: torch.dtype, layout: str = "agg") -> torch.Tensor:
    """``basis_compose``'s ``wn``: W_s = sum_b comp[live[s], b] basis[b] (fp32 fma chain, exact in budget), root as
    the last slab, rounded to op_dtype; layout "agg" [(S+1)*Fi, Fo], "tf" [Fi, (S+1)*Fo]."""
    w = _np64(weight)
    nb, fi, fo = w.shape
    if comp is None:
        c = np.eye(nb)[list(live)]
    else:
        c = _np64(comp)[list(live)]
    slabs = (c @ w.reshape(nb, -1)).reshape(len(live), fi, fo)
    abs_sum = (np.abs(c) @ np.abs(w).reshape(nb, -1)).reshape(len(live), fi, fo)
    check_budget(abs_sum, fraction_bits(c) + fraction_bits(w), what="basis_compose")
    if root is not None:
        slabs = np.concatenate([slabs, _np64(root)[None]], axis=0)
    s32 = _exact_f32(slabs, "basis_compose")
    out = round_to(s32, op_dtype)
    return out.reshape(-1, fo) if layout == "agg" else out.permute(1, 0, 2).reshape(fi, -1)


def expected_compose_bwd(weight: torch.Tensor, comp: torch.Tensor, dws: torch.Tensor, live: Sequence[int]):
    """(dweight [B, Fi, Fo], dcomp [R, B]) of ``basis_compose_bwd`` for the slab gradients ``dws`` [S, Fi, Fo]:
    dweight[b] = sum_s comp[live[s], b] dW_s and dcomp[live[s], b] = <dW_s, basis[b]> (fp32 partials, exact in
    budget); relations without a slot get exact zeros."""
    w = _np64(weight)
    nb, fi, fo = w.shape
    c = _np64(comp)
    d = _np64(dws).reshape(len(live), -1)
    cl = c[list(live)]
    dweight = cl.T @ d
    check_budget(np.abs(cl).T @ np.abs(d), fraction_bits(cl) + fraction_bits(d), what="basis_compose_bwd dweight")
    dc = d @ w.reshape(nb, -1).T
    check_budget(np.abs(d) @ np.abs(w).reshape(nb, -1).T, fraction_bits(d) + fraction_bits(w),
                 what="basis_compose_bwd dcomp")
    dcomp = np.zeros_like(c)
    dcomp[list(live)] = dc
    return (torch.from_numpy(_exact_f32(dweight, "dweight").reshape(nb, fi, fo)),
            torch.from_numpy(_exact_f32(dcomp, "dcomp")))
