"""The streaming normalisation kernels against plain fp64 references across their launch space:
GraphNorm and its column statistics (csrc/graphnorm.cu), LayerNorm (csrc/layernorm.cu) and soft
masking (csrc/graphnorm.cu).

The references are fp64 restatements run on the GPU: ``oracle.GraphNormRef`` (two-pass variance) with
``F.gelu`` where GELU is fused, ``torch.nn.LayerNorm``, ``oracle.soft_masking_ref`` and ``x.double()``
column sums; gradients come from autograd of the references.  The cases are picked to reach every
branch of the launch code: tiles narrower than a warp, threads that walk several rows (the unrolled
``kU`` loop), several column tiles, the 16-byte vector path and the scalar fallback (odd width,
misaligned base, leading dimension that is not a whole number of packs), and gradients that arrive as
``torch.cat`` views.  Data with a large offset against its spread, and constant columns, check the
one-pass variance where it cancels."""
import math

import pytest
import torch
import torch.nn.functional as F

import gmlm_b200 as G
from gmlm_b200 import ops
from oracle import GraphNormRef, soft_masking_ref

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5        # fp32 forward
FP32_GRAD_TOL = 2e-5   # fp32 gradients
BF16_TOL = 2e-2
EPS = 1e-5
K_MAX_ROW_BLOCKS = 148 * 8   # kMaxRowBlocks in graphnorm.cu: the most CTAs along the rows
K_U = 4                      # kU in graphnorm.cu: rows in flight per thread


def _rel(a: torch.Tensor, b: torch.Tensor, floor: float = 0.0) -> float:
    """conftest.rel_err (max |a-b| / max |b|) evaluated on the device: the large cases stay off the CPU."""
    a = a.detach().double()
    b = b.detach().double().to(a.device)
    if b.numel() == 0:
        return 0.0
    return float((a - b).abs().max() / b.abs().max().clamp(min=max(floor, 1e-30)))


def _gen(seed: int, dev) -> torch.Generator:
    return torch.Generator(device=dev).manual_seed(seed)


def _pack(dtype) -> int:
    return 16 // torch.tensor([], dtype=dtype).element_size()


LAYOUTS = ["contig", "slice", "misaligned", "odd_ld"]


def _place(t: torch.Tensor, layout: str, grad: bool = False) -> torch.Tensor:
    """``t`` as an [N, C] view of a fresh buffer in the given layout (``grad``: the buffer is a leaf that
    requires grad, so autograd reaches the view).  The rest of the buffer is NaN, so a read outside the view
    shows up in the result.
      contig      dense, ld = C
      slice       column slice at a 16-byte aligned offset, ld a multiple of the pack (vector path, ld != C)
      misaligned  column slice one element off a 16-byte boundary (scalar path)
      odd_ld      leading dimension that is not a multiple of the pack (scalar path)"""
    n, c = t.shape
    pack = _pack(t.dtype)
    if layout == "contig":
        return t.clone().requires_grad_(grad)
    if layout == "slice":
        ld, off = -(-c // pack) * pack + 2 * pack, pack
    elif layout == "misaligned":
        ld, off = -(-c // pack) * pack + 2 * pack, 1
    elif layout == "odd_ld":
        ld, off = (c + 1 if (c + 1) % pack else c + 2), 0
    else:
        raise ValueError(layout)
    buf = torch.full((n, ld), float("nan"), dtype=t.dtype, device=t.device)
    buf[:, off:off + c] = t
    v = buf.requires_grad_(grad)[:, off:off + c]
    assert v.stride() == (ld, 1)
    return v


def _vector_path(t: torch.Tensor) -> bool:
    """Mirror of vec_ok in graphnorm.cu for one operand."""
    pack = _pack(t.dtype)
    ld = t.stride(0) if t.size(0) > 1 else t.size(1)
    return t.size(1) % pack == 0 and t.data_ptr() % 16 == 0 and ld % pack == 0


def _rows_per_cta_pass(c: int, vec: int) -> int:
    """rpc of make_tile in graphnorm.cu: 256 threads, tpr (a power of two <= 256) of them along the row."""
    packs = -(-c // vec)
    tpr = 1
    while tpr < packs and tpr < 256:
        tpr <<= 1
    return 256 // tpr


def _gn_params(c: int, dev, seed: int, mean_scale_ones: bool = False):
    g = _gen(seed, dev)
    w = torch.rand(c, generator=g, device=dev) + 0.5
    b = torch.rand(c, generator=g, device=dev) - 0.5
    ms = torch.ones(c, device=dev) if mean_scale_ones else torch.rand(c, generator=g, device=dev) + 0.2
    return w, b, ms


def _gn_reference(x, gy, w, b, ms, fuse_gelu):
    """fp64 GraphNorm (+ exact GELU): output and the gradients of sum(y * gy) w.r.t. x, weight, bias, mean_scale."""
    c = x.size(1)
    ref = GraphNormRef(c).double().to(x.device)
    with torch.no_grad():
        ref.weight.copy_(w.double())
        ref.bias.copy_(b.double())
        ref.mean_scale.copy_(ms.double())
    x64 = x.detach().double().requires_grad_(True)
    y = ref(x64)
    if fuse_gelu:
        y = F.gelu(y)
    grads = torch.autograd.grad(y, (x64, ref.weight, ref.bias, ref.mean_scale), gy.double())
    return y.detach(), grads


def _gn_kernel(xv, gy, w, b, ms, fuse_gelu, cat_grad=False):
    """Forward and backward through the registered op.  ``cat_grad``: y goes through ``torch.cat`` with a
    3-wide block in front of it, so the backward receives gy as a narrow view (storage offset 3, ld C + 3)."""
    wl, bl, msl = (t.clone().requires_grad_(True) for t in (w, b, ms))
    y = G.graph_norm(xv, wl, bl, msl, EPS, fuse_gelu)
    if cat_grad:
        front = torch.zeros(y.size(0), 3, dtype=y.dtype, device=y.device)
        out = torch.cat([front, y], dim=1)
        gout = torch.cat([torch.randn_like(front), gy], dim=1)
        grads = torch.autograd.grad(out, (xv, wl, bl, msl), gout)
    else:
        grads = torch.autograd.grad(y, (xv, wl, bl, msl), gy)
    return y, grads


# ------------------------------------------------------------------ colstats
@pytest.mark.parametrize("n", [1, 4097, 300_001])
@pytest.mark.parametrize("c", [64, 37])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_colstats_exact(cuda_dev, n, c, dtype):
    """sum x and sum x^2 per column against fp64, for values about 1e3: fp32 input to 1e-12 (the squares
    and sums are fp64), bf16 to 1e-6 (per-thread running sums stay fp32 there by design)."""
    g = _gen(10 + n + c, cuda_dev)
    x = (1000.0 + 100.0 * torch.randn(n, c, generator=g, device=cuda_dev)).to(dtype)
    s, q = torch.ops.gmlm.colstats(x)
    assert s.dtype == q.dtype == torch.float64
    x64 = x.double()
    s64, q64 = x64.sum(0), x64.square().sum(0)
    tol = 1e-12 if dtype == torch.float32 else 1e-6
    assert float(((s - s64).abs() / s64.abs()).max()) <= tol
    assert float(((q - q64).abs() / q64).max()) <= tol


# ------------------------------------------------------------------ GraphNorm: constant columns
@pytest.mark.parametrize("n", [1000, 300_001])
def test_graph_norm_constant_columns(cuda_dev, n):
    """A bias-only or dead channel is a constant column: its variance is 0, so rstd = 1/sqrt(eps), y = bias,
    and the input gradient scales with that rstd.  Half the columns hold constants from U[1, 2000]."""
    c, half = 64, 32
    g = _gen(20 + n, cuda_dev)
    const = torch.rand(half, generator=g, device=cuda_dev) * 1999.0 + 1.0
    x = torch.empty(n, c, device=cuda_dev)
    x[:, :half] = const
    x[:, half:] = 3.0 + 2.0 * torch.randn(n, c - half, generator=g, device=cuda_dev)
    gy = torch.randn(n, c, generator=g, device=cuda_dev)
    w, b, ms = _gn_params(c, cuda_dev, 21, mean_scale_ones=True)

    y, mean, rstd = torch.ops.gmlm.graphnorm_fwd(x, w, b, ms, EPS, False)
    want_rstd = float(torch.tensor(1.0 / math.sqrt(float(torch.tensor(EPS, dtype=torch.float32))),
                                   dtype=torch.float32))
    assert float((rstd[:half].double() / want_rstd - 1.0).abs().max()) <= 1e-6
    assert torch.equal(mean[:half], const)
    assert _rel(y[:, :half], b[:half].expand(n, half)) <= FP32_TOL

    y_ref, (gx_r, gw_r, gb_r, gms_r) = _gn_reference(x, gy, w, b, ms, False)
    xl = x.clone().requires_grad_(True)
    y_k, (gx, gw, gb, gms) = _gn_kernel(xl, gy, w, b, ms, False)
    for cols in (slice(0, half), slice(half, c)):
        assert _rel(y_k[:, cols], y_ref[:, cols]) <= FP32_TOL
        assert _rel(gx[:, cols], gx_r[:, cols]) <= FP32_GRAD_TOL
        for got, want in ((gw, gw_r), (gb, gb_r), (gms, gms_r)):
            assert _rel(got[cols], want[cols]) <= FP32_GRAD_TOL


# ------------------------------------------------------------------ GraphNorm: offset sweep
@pytest.mark.parametrize("n", [183, 4097, 300_001])
@pytest.mark.parametrize("ms_ones", [True, False], ids=["a1", "a_rand"])
@pytest.mark.parametrize("sigma", [1.0, 1e-3])
@pytest.mark.parametrize("ratio", [0, 10, 100, 1000])
def test_graph_norm_offset(cuda_dev, ratio, sigma, ms_ones, n):
    """x = m + sigma * randn with m / sigma up to 1e3, fp32, forward and all four gradients.

    The forward stores the mean in fp32, and that rounding alone moves y by w * rstd * |shift error|,
    which near m / sigma = 1e3 and mean_scale = 1 reaches the 1e-5 gate by itself.  So every gate here is
    the suite's gate plus what storing the exact fp64 mean in fp32 costs each output (first-order, zero
    for m = 0), and the statistics themselves are pinned separately: the stored mean is the fp32 rounding
    of the fp64 mean and rstd matches fp64 to 1e-6."""
    c = 64
    g = _gen(int(ratio * 7 + n + (0 if ms_ones else 1) + (0 if sigma == 1.0 else 3)), cuda_dev)
    m = ratio * sigma
    x = (m + sigma * torch.randn(n, c, generator=g, device=cuda_dev)).float()
    gy = torch.randn(n, c, generator=g, device=cuda_dev)
    w, b, ms = _gn_params(c, cuda_dev, 30 + ratio, mean_scale_ones=ms_ones)

    x64 = x.double()
    mu64 = x64.mean(0)
    a64 = ms.double()
    rstd64 = 1.0 / ((x64 - mu64 * a64).square().mean(0) + float(torch.tensor(EPS, dtype=torch.float32))).sqrt()
    _, mean, rstd = torch.ops.gmlm.graphnorm_fwd(x, w, b, ms, EPS, False)
    assert float(((mean.double() - mu64).abs() - mu64.abs() * 2.0 ** -24).max()) <= 1e-12 * float(mu64.abs().max())
    assert float((rstd.double() / rstd64 - 1.0).abs().max()) <= 1e-6

    y_ref, (gx_r, gw_r, gb_r, gms_r) = _gn_reference(x, gy, w, b, ms, False)
    y, (gx, gw, gb, gms) = _gn_kernel(x.clone().requires_grad_(True), gy, w, b, ms, False)

    # |fl32(fl32(mu) * a) - mu * a|: the shift the kernels use, built from the exactly rounded mean
    shift = (mu64.float() * ms).double()
    dsh = (shift - mu64 * a64).abs()
    w64 = w.double().abs()
    floor_y = float((w64 * rstd64 * dsh).max() / y_ref.abs().max())
    floor_gw = float((rstd64 * dsh * gb_r.abs()).max() / gw_r.abs().max())
    floor_gx = float((w64 * rstd64.square() * dsh * gw_r.abs() / n).max() / gx_r.abs().max())
    floor_gms = float((mu64.square() * w64 * rstd64.pow(3) * (1 - a64).abs() * dsh * gb_r.abs()).max()
                      / gms_r.abs().max())
    assert _rel(y, y_ref) <= FP32_TOL + floor_y
    assert _rel(gx, gx_r) <= FP32_GRAD_TOL + floor_gx
    assert _rel(gw, gw_r) <= FP32_GRAD_TOL + floor_gw
    assert _rel(gb, gb_r) <= FP32_GRAD_TOL
    assert _rel(gms, gms_r) <= FP32_GRAD_TOL + floor_gms


# ------------------------------------------------------------------ GraphNorm: launch space
GN_SHAPES = [
    (1, 8), (2, 4), (7, 3),               # tiny tiles
    (183, 16),                            # tpr < 32
    (300_001, 64), (20_000, 512),         # several rows per thread: the kU loop is live
    (5000, 1703), (3000, 4096),           # several column tiles (1703: scalar in fp32)
]
MULTI_ROW = {(300_001, 64), (20_000, 512)}


@pytest.mark.parametrize("layout", LAYOUTS + ["cat_grad"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("fuse_gelu", [False, True], ids=["plain", "gelu"])
@pytest.mark.parametrize("n,c", GN_SHAPES)
def test_graph_norm_launch_space(cuda_dev, n, c, fuse_gelu, dtype, layout):
    g = _gen(n * 31 + c, cuda_dev)
    x = (3.0 + 2.0 * torch.randn(n, c, generator=g, device=cuda_dev)).to(dtype)
    gy = torch.randn(n, c, generator=g, device=cuda_dev).to(dtype)
    w, b, ms = _gn_params(c, cuda_dev, 40 + c)
    xv = _place(x, "contig" if layout == "cat_grad" else layout, grad=True)
    gyv = gy if layout == "cat_grad" else _place(gy, layout)
    if layout in ("contig", "slice", "cat_grad") and c % _pack(dtype) == 0:
        assert _vector_path(xv)
    if layout in ("misaligned", "odd_ld") and n > 1:
        assert not _vector_path(xv)
    if (n, c) in MULTI_ROW:
        # the vector path has the most rows per CTA pass: a thread sees a second kU group on either path
        rpc = _rows_per_cta_pass(c, _pack(dtype) if c % _pack(dtype) == 0 else 1)
        assert n > K_MAX_ROW_BLOCKS * rpc * K_U

    y_ref, grads_ref = _gn_reference(x, gy, w, b, ms, fuse_gelu)
    y, grads = _gn_kernel(xv, gyv, w, b, ms, fuse_gelu, cat_grad=(layout == "cat_grad"))
    assert y.dtype == dtype and grads[0].dtype == dtype
    fwd_tol, grad_tol = (FP32_TOL, FP32_GRAD_TOL) if dtype == torch.float32 else (BF16_TOL, BF16_TOL)
    assert _rel(y, y_ref) <= fwd_tol
    floors = {}
    if n == 1:
        # One row: ohat^2 = 1 - eps*rstd^2, so gx = w*rstd*dn*(1 - ohat^2) - ... and gms = -mu*w*rstd*dn*(1 - ohat^2)
        # are ~1e-6 of the terms they are formed from, and both sides of the comparison are mostly rounding.
        # Those two are gated against the size of the terms (rel_err's floor).  (The encoder skips GraphNorm
        # on a single node.)
        x64 = x.double()
        rstd64 = ((x64 - x64 * ms.double()).square() + EPS).rsqrt()
        terms = (w.double() * rstd64 * gy.double()).abs()
        floors = {"gx": float(terms.max()), "gms": float((x64.abs() * terms).max())}
    for name, got, want in zip(("gx", "gw", "gb", "gms"), grads, grads_ref):
        assert _rel(got, want, floor=floors.get(name, 0.0)) <= grad_tol, name


# ------------------------------------------------------------------ GraphNorm: partitioned statistics
@pytest.mark.parametrize("k", [2, 3])
@pytest.mark.parametrize("fuse_gelu", [False, True], ids=["plain", "gelu"])
def test_graph_norm_partitioned_stats(cuda_dev, k, fuse_gelu):
    """The arithmetic of dist_norm.py on one GPU, without the collectives: per-slice colstats summed, the
    forward applied per slice with stat_rows = N; per-slice backward sums summed, the backward applied per
    slice.  k non-empty slices plus an empty one."""
    n, c = 50_001, 96
    g = _gen(50 + k, cuda_dev)
    x = 3.0 + 2.0 * torch.randn(n, c, generator=g, device=cuda_dev)
    gy = torch.randn(n, c, generator=g, device=cuda_dev)
    w, b, ms = _gn_params(c, cuda_dev, 51)
    cuts = [0] + [n * i // k + 17 * i for i in range(1, k)] + [n]
    bounds = list(zip(cuts[:-1], cuts[1:]))
    bounds.insert(1, (cuts[1], cuts[1]))                  # an empty slice
    parts = [x[lo:hi] for lo, hi in bounds]
    gparts = [gy[lo:hi] for lo, hi in bounds]
    assert sum(p.size(0) for p in parts) == n and any(p.size(0) == 0 for p in parts)

    stats = [torch.ops.gmlm.colstats(p) for p in parts]
    s = sum(t[0] for t in stats)
    q = sum(t[1] for t in stats)
    fw = [ops.graphnorm_apply_stats(p, s, q, w, b, ms, EPS, fuse_gelu, stat_rows=n) for p in parts]
    mean, rstd = fw[0][1], fw[0][2]
    for _, m_i, r_i in fw:
        assert torch.equal(m_i, mean) and torch.equal(r_i, rstd)
    bs = [ops.graphnorm_bwd_stats(p, gp, mean, rstd, w, b, ms, fuse_gelu) for p, gp in zip(parts, gparts)]
    s1 = sum(t[0] for t in bs)
    s2 = sum(t[1] for t in bs)
    bw = [ops.graphnorm_bwd_apply(p, gp, mean, rstd, w, b, ms, fuse_gelu, s1, s2, True, stat_rows=n)
          for p, gp in zip(parts, gparts)]

    y_ref, (gx_r, gw_r, gb_r, gms_r) = _gn_reference(x, gy, w, b, ms, fuse_gelu)
    assert _rel(torch.cat([t[0] for t in fw]), y_ref) <= FP32_TOL
    assert _rel(torch.cat([t[0] for t in bw]), gx_r) <= FP32_GRAD_TOL
    for i, want in ((1, gw_r), (2, gb_r), (3, gms_r)):
        for t in bw:
            assert torch.equal(t[i], bw[0][i])
        assert _rel(bw[0][i], want) <= FP32_GRAD_TOL


# ------------------------------------------------------------------ determinism
def test_reductions_deterministic(cuda_dev):
    """Every column / parameter reduction is order-fixed: two calls give identical bits."""
    n, c = 300_001, 64
    g = _gen(60, cuda_dev)
    x = 3.0 + 2.0 * torch.randn(n, c, generator=g, device=cuda_dev)
    gy = torch.randn(n, c, generator=g, device=cuda_dev)
    a, b_ = torch.ops.gmlm.colstats(x), torch.ops.gmlm.colstats(x)
    assert torch.equal(a[0], b_[0]) and torch.equal(a[1], b_[1])

    w, b, ms = _gn_params(c, cuda_dev, 61)
    r1 = _gn_kernel(x.clone().requires_grad_(True), gy, w, b, ms, True)[1]
    r2 = _gn_kernel(x.clone().requires_grad_(True), gy, w, b, ms, True)[1]
    for u, v in zip(r1[1:], r2[1:]):
        assert torch.equal(u, v)

    lw, lb = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    l1 = torch.autograd.grad(G.layer_norm(x, lw, lb), (lw, lb), gy)
    l2 = torch.autograd.grad(G.layer_norm(x, lw, lb), (lw, lb), gy)
    assert torch.equal(l1[0], l2[0]) and torch.equal(l1[1], l2[1])

    mask = torch.rand(n, generator=g, device=cuda_dev) < 0.3
    tok = torch.randn(1, c, generator=g, device=cuda_dev).requires_grad_(True)
    t1 = torch.autograd.grad(G.soft_masking_gnn_input(x, mask, tok), tok, gy)[0]
    t2 = torch.autograd.grad(G.soft_masking_gnn_input(x, mask, tok), tok, gy)[0]
    assert torch.equal(t1, t2)


# ------------------------------------------------------------------ LayerNorm
def _ln_reference(x, gy, w, b):
    c = x.size(1)
    ref = torch.nn.LayerNorm(c).double().to(x.device)
    with torch.no_grad():
        ref.weight.copy_(w.double())
        ref.bias.copy_(b.double())
    x64 = x.detach().double().requires_grad_(True)
    y = ref(x64)
    return y.detach(), torch.autograd.grad(y, (x64, ref.weight, ref.bias), gy.double())


def _ln_kernel(xv, gy, w, b):
    wl, bl = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    y = G.layer_norm(xv, wl, bl, EPS)
    return y, torch.autograd.grad(y, (xv, wl, bl), gy)


def _ln_params(c, dev, seed):
    g = _gen(seed, dev)
    return torch.rand(c, generator=g, device=dev) + 0.5, torch.rand(c, generator=g, device=dev) - 0.5


def _ln_check(x, gy, w, b, xv=None, gyv=None):
    y_ref, grads_ref = _ln_reference(x, gy, w, b)
    if xv is None:
        xv = x.clone().requires_grad_(True)
    y, grads = _ln_kernel(xv, gy if gyv is None else gyv, w, b)
    tol, gtol = (FP32_TOL, FP32_GRAD_TOL) if x.dtype == torch.float32 else (BF16_TOL, BF16_TOL)
    assert y.dtype == x.dtype
    assert _rel(y, y_ref) <= tol
    for name, got, want in zip(("gx", "ggamma", "gbeta"), grads, grads_ref):
        assert _rel(got, want) <= gtol, name


# fp32 NP = 1, 2, 4, 6, 8 (NP = packs of 4 per lane) and bf16 NP = 1, 2, 3, 4 (packs of 8)
LN_WIDTHS = ([(torch.float32, c) for c in (4, 128, 132, 256, 260, 512, 516, 768, 772, 1024)] +
             [(torch.bfloat16, c) for c in (8, 256, 264, 512, 520, 768, 776, 1024)])


@pytest.mark.parametrize("n", [1, 9, 4097])
@pytest.mark.parametrize("dtype,c", LN_WIDTHS, ids=[f"{'f32' if d == torch.float32 else 'bf16'}-{c}"
                                                    for d, c in LN_WIDTHS])
def test_layer_norm_template_widths(cuda_dev, dtype, c, n):
    g = _gen(70 + c + n, cuda_dev)
    x = (3.0 + 2.0 * torch.randn(n, c, generator=g, device=cuda_dev)).to(dtype)
    gy = torch.randn(n, c, generator=g, device=cuda_dev).to(dtype)
    w, b = _ln_params(c, cuda_dev, 71)
    _ln_check(x, gy, w, b)


@pytest.mark.parametrize("dtype,c", [(torch.float32, 128), (torch.bfloat16, 256)], ids=["f32", "bf16"])
def test_layer_norm_many_rows_per_warp(cuda_dev, dtype, c):
    """N = 1 000 003: each warp walks hundreds of rows, so the per-lane fp32 gamma/beta partials are long sums."""
    n = 1_000_003
    g = _gen(72, cuda_dev)
    x = (3.0 + 2.0 * torch.randn(n, c, generator=g, device=cuda_dev)).to(dtype)
    gy = torch.randn(n, c, generator=g, device=cuda_dev).to(dtype)
    w, b = _ln_params(c, cuda_dev, 73)
    _ln_check(x, gy, w, b)


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("dtype,c", [(torch.float32, 256), (torch.float32, 8), (torch.bfloat16, 768)],
                         ids=["f32-256", "f32-8", "bf16-768"])
def test_layer_norm_views(cuda_dev, dtype, c, layout):
    """Inputs and incoming gradients that are views: an aligned column slice runs in place, a view the
    kernel cannot read in 16-byte packs is copied first; all must match the reference."""
    n = 1000
    g = _gen(80 + c, cuda_dev)
    x = (3.0 + 2.0 * torch.randn(n, c, generator=g, device=cuda_dev)).to(dtype)
    gy = torch.randn(n, c, generator=g, device=cuda_dev).to(dtype)
    w, b = _ln_params(c, cuda_dev, 81)
    xv = _place(x, layout, grad=True)
    assert ops.layer_norm_ok(xv)
    _ln_check(x, gy, w, b, xv=xv, gyv=_place(gy, layout))


@pytest.mark.parametrize("width", [3, 8])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_layer_norm_cat_backward(cuda_dev, dtype, width):
    """torch.cat([other, layer_norm(x)], 1).backward(): the LayerNorm backward receives gy as a narrow
    view (storage offset = width of `other`, ld = C + width)."""
    n, c = 777, 64
    g = _gen(90 + width, cuda_dev)
    x = torch.randn(n, c, generator=g, device=cuda_dev).to(dtype)
    other = torch.randn(n, width, generator=g, device=cuda_dev).to(dtype).requires_grad_(True)
    gout = torch.randn(n, width + c, generator=g, device=cuda_dev).to(dtype)
    w, b = _ln_params(c, cuda_dev, 91)
    xl, wl, bl = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    torch.cat([other, G.layer_norm(xl, wl, bl, EPS)], dim=1).backward(gout)
    _, (gx_r, gw_r, gb_r) = _ln_reference(x, gout[:, width:], w, b)
    gtol = FP32_GRAD_TOL if dtype == torch.float32 else BF16_TOL
    assert _rel(xl.grad, gx_r) <= gtol
    assert _rel(wl.grad, gw_r) <= gtol
    assert _rel(bl.grad, gb_r) <= gtol
    assert torch.equal(other.grad, gout[:, :width])


@pytest.mark.parametrize("m", [0.0, 100.0, 1000.0])
def test_layer_norm_row_offset(cuda_dev, m):
    """Rows with mean m and unit spread.  The kernel's row mean is an fp32 warp sum, as the stock op's is,
    so the gate is relative to the stock op: error vs fp64 <= max(suite gate, 2 x torch.nn.LayerNorm fp32)."""
    n, c = 4097, 256
    g = _gen(100 + int(m), cuda_dev)
    x = m + torch.randn(n, c, generator=g, device=cuda_dev)
    gy = torch.randn(n, c, generator=g, device=cuda_dev)
    w, b = _ln_params(c, cuda_dev, 101)
    y_ref, grads_ref = _ln_reference(x, gy, w, b)
    stock = torch.nn.LayerNorm(c).to(cuda_dev)
    with torch.no_grad():
        stock.weight.copy_(w)
        stock.bias.copy_(b)
    xs = x.clone().requires_grad_(True)
    ys = stock(xs)
    gs = torch.autograd.grad(ys, (xs, stock.weight, stock.bias), gy)
    y, grads = _ln_kernel(x.clone().requires_grad_(True), gy, w, b)
    assert _rel(y, y_ref) <= max(FP32_TOL, 2 * _rel(ys, y_ref))
    for name, got, st, want in zip(("gx", "ggamma", "gbeta"), grads, gs, grads_ref):
        assert _rel(got, want) <= max(FP32_GRAD_TOL, 2 * _rel(st, want)), name


# ------------------------------------------------------------------ soft masking
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("ratio", [0.0, 0.3, 1.0])
@pytest.mark.parametrize("n", [0, 1, 300_001])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_soft_mask(cuda_dev, dtype, n, ratio, layout):
    """fp32: bit-exact to the reference's rounding sequence on every layout.  bf16: within one bf16 rounding
    of the fp64 result.  g_token (beta * masked column sum of gy) against fp64."""
    f, beta = 96, 0.7
    g = _gen(110 + n + int(ratio * 10), cuda_dev)
    x = torch.randn(n, f, generator=g, device=cuda_dev).to(dtype)
    gy = torch.randn(n, f, generator=g, device=cuda_dev).to(dtype)
    mask = torch.rand(n, generator=g, device=cuda_dev) < ratio
    token = (torch.randn(1, f, generator=g, device=cuda_dev) * 0.1)
    xv = _place(x, layout)
    tok = token.clone().requires_grad_(True)
    y = G.soft_masking_gnn_input(xv, mask, tok, beta=beta)
    assert y.dtype == dtype and y.shape == (n, f)
    g_tok, = torch.autograd.grad(y, tok, _place(gy, layout))

    m = mask.unsqueeze(1)
    x64, t64 = x.double(), token.double()
    y64 = torch.where(m, (1 - beta) * x64 + beta * t64, x64)
    gtok64 = beta * (gy.double() * m).sum(0, keepdim=True)
    if dtype == torch.float32:
        assert torch.equal(y, soft_masking_ref(x, mask, token, beta=beta))
    else:
        assert torch.equal(y[~mask], x[~mask])
        # one rounding to bf16 (relative 2^-8) of a value computed in fp32 (absolute 2^-22 of the terms)
        bound = y64.abs() * 2.0 ** -8 + ((1 - beta) * x64.abs() + beta * t64.abs()) * 2.0 ** -22
        assert bool(((y.double() - y64).abs() <= bound).all())
    if n == 0 or ratio == 0.0:
        assert torch.count_nonzero(g_tok) == 0
    else:
        assert _rel(g_tok, gtok64) <= (FP32_TOL if dtype == torch.float32 else BF16_TOL)

    # input gradient: (1 - beta) * gy on masked rows, gy elsewhere
    xl = _place(x, layout, grad=True)
    gx, = torch.autograd.grad(G.soft_masking_gnn_input(xl, mask, token, beta=beta), xl, _place(gy, layout))
    gx64 = torch.where(m, (1 - beta) * gy.double(), gy.double())
    assert torch.equal(gx[~mask], gy[~mask])
    if dtype == torch.float32:
        assert _rel(gx, gx64) <= FP32_TOL
    else:
        assert bool(((gx.double() - gx64).abs() <= gx64.abs() * 2.0 ** -8 + gy.double().abs() * 2.0 ** -22).all())
