"""The dense kernels bit for bit on integer operands (csrc/gemm_tcgen05.cu, csrc/compose.cu): ``gemm_nt`` on bf16 /
fp16 and on fp32 (3xTF32) operands with its bias, addend, split and routed outputs, ``gemm_tn`` with every split
boundary of a 300k-row reduction, and the basis composition forward and backward across their launch loops.
Products of small integers and dyadic coefficients are exact and their sums stay exact in fp32 (under 2^22 units
on the tensor cores), so each output is fixed up to its epilogue, which ``exact_arith`` reproduces."""
import pytest
import torch

from gmlm_b200.ops import basis_compose, basis_compose_bwd, gemm_nt, gemm_tn

import exact_arith as X

pytestmark = pytest.mark.gpu


def _ints(shape, dtype, seed, **kw):
    return X.int_tensor(shape, dtype, seed=seed, device="cuda", **kw)


# ------------------------------------------------------------------------------ gemm_nt
@pytest.mark.parametrize("op", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("m,n,ks", [(128, 64, (64,)), (389, 256, (64,)), (1000, 128, (256, 64)), (77, 32, (192,)),
                                    (5, 96, (64,)), (30011, 1280, (64,)), (300, 512, (1200, 300)),
                                    (129, 36, (70, 30, 20)), (5000, 768, (64, 128, 256, 512)), (999, 200, (72, 200)),
                                    (257, 1500, (512,)), (64, 8, (8,))])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
def test_gemm_nt_exact(cuda_dev, op, m, n, ks, out_dtype):
    """Ragged M / N / K, partial last k-blocks of one to four sources, a dyadic bias."""
    seed = m + n + sum(ks)
    srcs = [_ints((m, k), op, seed + i) for i, k in enumerate(ks)]
    b = _ints((n, sum(ks)), op, seed + 7)
    bias = X.dyadic_weights(n, seed=seed, device="cuda")
    got = gemm_nt(srcs, b, bias=bias, out_dtype=out_dtype)
    assert got.dtype == out_dtype
    assert torch.equal(got.cpu(), X.expected_gemm(srcs, b, bias=bias, out_dtype=out_dtype))


@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("m,n,k", [(1000, 512, 300), (4099, 64, 256), (70, 128, 64), (2500, 1024, 512)])
def test_gemm_nt_addend_exact(cuda_dev, m, n, k, out_dtype):
    """C = A B^T + bias + addend in fp32, ONE rounding: a bf16 store of A B^T + bias before the addend differs."""
    a = _ints((m, k), torch.bfloat16, k)
    b = _ints((n, k), torch.bfloat16, k + 1)
    bias = X.dyadic_weights(n, seed=k, device="cuda")
    add = _ints((m, n), out_dtype, k + 2, lo=-64, hi=64)
    got = gemm_nt(a, b, bias=bias, out_dtype=out_dtype, addend=add)
    assert torch.equal(got.cpu(), X.expected_gemm(a, b, bias=bias, addend=add, out_dtype=out_dtype))


@pytest.mark.parametrize("op", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("widths", [(1024, 256), (1200, 300), (30, 300), (64, 128, 256, 512), (128, 64, 40),
                                    (256, 256, 256, 192)])
def test_gemm_nt_split_and_routed_outputs_exact(cuda_dev, op, widths):
    m, k = 3001, 768
    a = _ints((m, k), op, sum(widths))
    b = _ints((sum(widths), k), op, len(widths))
    outs = gemm_nt(a, b, out_dtype=torch.float32, split=widths[0] if len(widths) == 2 else list(widths))
    want = X.expected_gemm(a, b)
    c0 = 0
    for o, w in zip(outs, widths):
        assert torch.equal(o.cpu(), want[:, c0:c0 + w])
        c0 += w


@pytest.mark.parametrize("m,n,ks", [(300, 512, (1200, 300)), (1000, 100, (100,)), (777, 36, (72, 20)), (64, 8, (4,)),
                                    (9000, 320, (1703,)), (4097, 64, (1024, 256))])
@pytest.mark.parametrize("use_bias", [False, True])
def test_gemm_nt_fp32_3xtf32_exact(cuda_dev, m, n, ks, use_bias):
    """fp32 integer operands: the hi parts carry them whole, the lo parts are zero -- tiling, k-blocks and source
    routing of the 3xTF32 kernel pinned bit for bit (its hi/lo accuracy is the fp64 test's)."""
    seed = m + n
    srcs = [_ints((m, k), torch.float32, seed + i) for i, k in enumerate(ks)]
    b = _ints((n, sum(ks)), torch.float32, seed + 9)
    bias = X.dyadic_weights(n, seed=seed, device="cuda") if use_bias else None
    got = gemm_nt(srcs, b, bias=bias)
    assert torch.equal(got.cpu(), X.expected_gemm(srcs, b, bias=bias))
    c1, c2 = gemm_nt(srcs, b, bias=bias, split=n // 3 or 1)
    assert torch.equal(torch.cat([c1, c2], 1).cpu(), X.expected_gemm(srcs, b, bias=bias))


# ------------------------------------------------------------------------------ gemm_tn
@pytest.mark.parametrize("op", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("m,ks,n", [(1000, (64,), 64), (100000, (256, 64), 64), (5000, (1200, 300), 512),
                                    (70000, (256,), 320), (777, (100, 36), 200), (30000, (64, 128, 256, 512), 96),
                                    (200, (8,), 8), (37, (130,), 70), (300000, (128,), 64)])
def test_gemm_tn_exact(cuda_dev, op, m, ks, n):
    """Operands without zeros: a row dropped or added at a split boundary, or a split left out of the final sum,
    changes the result by at least 1."""
    seed = m + n
    srcs = [_ints((m, k), op, seed + i, lo=-2, hi=2, nonzero=True) for i, k in enumerate(ks)]
    g = _ints((m, n), op, seed + 5, lo=-2, hi=2, nonzero=True)
    got = gemm_tn(srcs, g)
    assert torch.equal(got.cpu(), X.expected_gemm_tn(srcs, g))


# ------------------------------------------------------------------------------ basis composition
def _compose_params(nb, r, fi, fo, seed):
    weight = _ints((nb, fi, fo), torch.float32, seed)
    comp = X.dyadic_weights((r, nb), seed=seed + 1, device="cuda")
    root = _ints((fi, fo), torch.float32, seed + 2)
    return weight, comp, root


LIVE = {1: (3,), 4: (0, 1, 2, 3), 5: (4, 0, 2, 6, 1), 8: tuple(range(1, 9)), 9: (0, 2, 3, 5, 6, 7, 9, 10, 11),
        12: tuple(range(12))}


@pytest.mark.parametrize("op", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("layout", ["agg", "tf"])
@pytest.mark.parametrize("S,nb,fi,fo", [(1, 30, 64, 64), (4, 33, 300, 512), (5, 70, 33, 20), (8, 1, 100, 7),
                                        (9, 30, 257, 36), (12, 33, 17, 22), (12, 70, 48, 64)])
def test_basis_compose_exact(cuda_dev, op, layout, S, nb, fi, fo):
    """Both MAXS instances (S <= 4, <= 8), the multi-launch loop over slots (S > 8), Fo on 4-wide and scalar packs,
    ragged Fi."""
    live = LIVE[S]
    weight, comp, root = _compose_params(nb, 13, fi, fo, S * 100 + nb)
    wn, wt = basis_compose(weight, comp, root, live, op, layout)
    want = X.expected_compose(weight, comp, root, live, op, layout)
    assert torch.equal(wn.cpu(), want) and torch.equal(wt.cpu(), want.t())


@pytest.mark.parametrize("S", [4, 9])
@pytest.mark.parametrize("layout", ["agg", "tf"])
def test_basis_compose_without_comp_or_root_exact(cuda_dev, S, layout):
    live = LIVE[S]
    weight, comp, root = _compose_params(13, 13, 40, 24, S)
    for c, r in ((None, root), (comp, None), (None, None)):
        wn, wt = basis_compose(weight, c, r, live, torch.bfloat16, layout)
        want = X.expected_compose(weight, c, r, live, torch.bfloat16, layout)
        assert torch.equal(wn.cpu(), want) and torch.equal(wt.cpu(), want.t())


@pytest.mark.parametrize("nb", [1, 30, 33, 70])
@pytest.mark.parametrize("r,live", [(5, (0, 1, 2, 3)), (64, (63, 0, 17, 5, 40, 2, 33, 61)), (13, (2,))])
@pytest.mark.parametrize("layout", ["agg", "tf"])
def test_basis_compose_bwd_exact(cuda_dev, nb, r, live, layout):
    """dweight and dcomp bit for bit: bases past 32 (the second launch over bases), 64 relations with 8 live ones
    (the kernel's limits), relations without a slot exactly zero."""
    fi, fo = 100, 36
    S = len(live)
    weight, comp, _ = _compose_params(nb, r, fi, fo, nb + r)
    dws = _ints((S, fi, fo), torch.float32, nb * r)
    if layout == "agg":
        dw, ss, rs = dws.contiguous(), fi * fo, fo
    else:
        dw = torch.cat([dws.permute(1, 0, 2).reshape(fi, S * fo), torch.zeros(fi, fo, device="cuda")], 1).contiguous()
        ss, rs = fo, (S + 1) * fo
    dweight, dcomp = basis_compose_bwd(weight, comp, dw, ss, rs, live)
    want_w, want_c = X.expected_compose_bwd(weight, comp, dws, live)
    assert torch.equal(dweight.cpu(), want_w) and torch.equal(dcomp.cpu(), want_c)


@pytest.mark.parametrize("S,fo", [(9, 36), (4, 22), (12, 7)])
def test_basis_compose_bwd_torch_shapes_exact(cuda_dev, S, fo):
    """More than 8 populated relations or Fo % 4 != 0: the two fp32 matmuls outside the kernel, exact as well."""
    live = LIVE[S]
    nb, fi = 33, 50
    weight, comp, _ = _compose_params(nb, 13, fi, fo, S + fo)
    dws = _ints((S, fi, fo), torch.float32, S * fo)
    dweight, dcomp = basis_compose_bwd(weight, comp, dws.contiguous(), fi * fo, fo, live)
    want_w, want_c = X.expected_compose_bwd(weight, comp, dws, live)
    assert torch.equal(dweight.cpu(), want_w) and torch.equal(dcomp.cpu(), want_c)
