"""The exact-arithmetic references of ``exact_arith`` against step-by-step numpy float32, on the CPU: the predicted
mean and rounding (ties to even in bf16 and fp16 included), and the budget asserts that keep a reference from
predicting a value the kernels cannot compute exactly."""
import numpy as np
import pytest
import torch

import exact_arith as X


def _step_by_step(x32, rowptr, col, w, mode, rng):
    """One fp32 add (or fma) at a time, edges in a random order per row, then the mean's fp32 scale."""
    out = np.zeros((rowptr.size - 1, x32.shape[1]), np.float32)
    for r in range(rowptr.size - 1):
        es = rng.permutation(np.arange(rowptr[r], rowptr[r + 1]))
        acc = np.zeros(x32.shape[1], np.float32)
        for e in es:
            term = x32[col[e]] * (w[e] if mode == X.AGG_WEIGHTED else np.float32(1))
            acc = (acc + term).astype(np.float32)
        L = rowptr[r + 1] - rowptr[r]
        if mode == X.AGG_MEAN and L > 1:
            acc = acc * (np.float32(1) / np.float32(L))
        out[r] = acc
    return out


@pytest.mark.parametrize("mode", [X.AGG_SUM, X.AGG_MEAN, X.AGG_WEIGHTED])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_expected_spmm_matches_step_by_step_fp32(mode, dtype):
    rng = np.random.default_rng(mode * 7 + (dtype == torch.bfloat16))
    n_rows, n_src, feat = 60, 40, 12
    lens = rng.choice([0, 1, 2, 3, 5, 7, 64, 100, 300], size=n_rows)
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = rng.integers(0, n_src, rowptr[-1])
    x = X.int_tensor((n_src, feat), dtype, seed=3)
    w = X.dyadic_weights(rowptr[-1], seed=4)
    got = X.expected_spmm(x, rowptr, col, mode, w if mode == X.AGG_WEIGHTED else None)
    ref32 = _step_by_step(x.float().numpy(), rowptr, col, w.numpy(), mode, rng)
    assert got.dtype == dtype
    assert torch.equal(got, torch.from_numpy(ref32).to(dtype))     # torch's own fp32 -> bf16 is round-to-nearest-even


def test_expected_spmm_per_head_weights():
    rowptr = np.array([0, 3, 3, 5])
    col = np.array([0, 1, 1, 2, 0])
    x = torch.tensor([[1., 2., 3., 4.], [-1., 0., 2., 1.], [4., 4., -4., 1.]])
    w = torch.tensor([[1., 2.], [0.5, 0.25], [-2., 1.], [1., 1.], [0.25, -1.]])
    got = X.expected_spmm(x, rowptr, col, X.AGG_WEIGHTED, w)
    want = torch.tensor([[1 - 0.5 + 2, 2 + 0 - 0, 2 * 3 + 0.25 * 2 + 2, 2 * 4 + 0.25 + 1],
                         [0, 0, 0, 0],
                         [4 + 0.25, 4 + 0.5, -4 - 3, 1 - 4]])
    assert torch.equal(got, want)


def test_round_to_ties_to_even():
    # bf16 keeps 7 fraction bits: 1 + 2^-8 is a tie between 1 and 1 + 2^-7 (-> 1), 1 + 3 * 2^-8 one between
    # 1 + 2^-7 and 1 + 2^-6 (-> 1 + 2^-6); truncation would give 1 and 1 + 2^-7
    v = np.array([1 + 2 ** -8, 1 + 3 * 2 ** -8, -(1 + 3 * 2 ** -8), 257, 259, 1 + 2 ** -8 + 2 ** -20], np.float32)
    assert X.round_to(v, torch.bfloat16).float().tolist() == [1.0, 1 + 2 ** -6, -(1 + 2 ** -6), 256, 260, 1 + 2 ** -7]
    # fp16 keeps 10: 1 + 2^-11 -> 1, 1 + 3 * 2^-11 -> 1 + 2^-9, 2049 -> 2048, 2051 -> 2052
    v = np.array([1 + 2 ** -11, 1 + 3 * 2 ** -11, 2049, 2051], np.float32)
    assert X.round_to(v, torch.float16).float().tolist() == [1.0, 1 + 2 ** -9, 2048, 2052]
    rng = np.random.default_rng(0)
    r = (rng.standard_normal(100_000) * 1000).astype(np.float32)
    assert torch.equal(X.round_to(r, torch.bfloat16), torch.from_numpy(r).bfloat16())
    assert torch.equal(X.round_to(r, torch.float16), torch.from_numpy(r).half())


def test_mean_of_a_tie_rounds_to_even():
    """S / L exact in fp32 but halfway between two bf16 numbers: 257 / 256 -> 1, 259 / 256 -> 1 + 2^-6."""
    rowptr = np.array([0, 256, 512])
    col = np.zeros(512, np.int64)
    x = torch.ones(1, 1)
    w = torch.ones(512)
    w[0], w[256] = 2.0, 4.0                               # row sums 257 and 259
    s = X.expected_spmm(x, rowptr, col, X.AGG_WEIGHTED, w)
    assert s.flatten().tolist() == [257.0, 259.0]
    xb = torch.tensor([[1.0], [2.0], [4.0]]).bfloat16()
    col = np.zeros(512, np.int64)
    col[0], col[256] = 1, 2                               # the same sums as a mean over 256 edges
    m = X.expected_spmm(xb, rowptr, col, X.AGG_MEAN)
    assert m.float().flatten().tolist() == [1.0, 1 + 2 ** -6]


def test_mean_scale_is_the_fp32_reciprocal():
    """L = 7: the kernels multiply by fp32(1/7), not divide by 7 -- for S = 7 * 3 the two differ."""
    rowptr = np.array([0, 7])
    col = np.zeros(7, np.int64)
    x = torch.full((1, 1), 3.0)
    got = X.expected_spmm(x, rowptr, col, X.AGG_MEAN).item()
    assert got == float(np.float32(21) * (np.float32(1) / np.float32(7)))
    assert got != 3.0


def test_budget_asserts_fire():
    # 2^20 edges of |x| = 16 in one row: 2^24, one unit past the exact range
    rowptr = np.array([0, 1 << 20])
    col = np.zeros(1 << 20, np.int64)
    with pytest.raises(AssertionError, match="exact range"):
        X.expected_spmm(torch.full((1, 1), 16.0), rowptr, col, X.AGG_SUM)
    X.expected_spmm(torch.full((1, 1), 15.0), rowptr, col, X.AGG_SUM)
    # weights of 1/4 count in units of 2^-2: the same row at |x| = 4 and w = 1/4 is 2^20 * 2^2 = 2^22 units: fine;
    # 2^22 of them are 2^24: out
    w = torch.full((1 << 20,), 0.25)
    X.expected_spmm(torch.full((1, 1), 4.0), rowptr, col, X.AGG_WEIGHTED, w)
    with pytest.raises(AssertionError, match="exact range"):
        X.expected_spmm(torch.full((1, 1), 16.0), rowptr, col, X.AGG_WEIGHTED, w)
    # weights that are not short dyadic fractions count in units of their last fp32 bit: fp32(1/3) is a multiple
    # of 2^-25, so four such terms already leave the range
    with pytest.raises(AssertionError, match="exact range"):
        X.expected_spmm(torch.ones(1, 1), np.array([0, 4]), np.zeros(4, np.int64), X.AGG_WEIGHTED,
                        torch.full((4,), 1 / 3))
    # tensor-core products: 2^22 units
    a = torch.full((1, 1 << 18), 4.0)
    with pytest.raises(AssertionError, match="exact range"):
        X.expected_gemm(a, a.clone())
    X.expected_gemm(a[:, :(1 << 18) - 1], a[:, :(1 << 18) - 1])
    with pytest.raises(AssertionError, match="exact range"):
        X.expected_gemm_tn(torch.full((1 << 20, 1), 2.0), torch.full((1 << 20, 1), 2.0))
    # composition: an fp32 fma chain over the bases
    basis = torch.full((4, 1, 1), 2.0 ** 21)
    with pytest.raises(AssertionError, match="exact range"):
        X.expected_compose(basis, torch.full((1, 4), 2.0), None, [0], torch.float32)
    with pytest.raises(AssertionError, match="exact range"):
        X.expected_compose_bwd(basis, torch.full((1, 4), 2.0), torch.full((1, 1, 1), 8.0), [0])


def test_expected_dense_epilogue_order():
    """bias first, then the addend, each an fp32 add, one rounding: (acc + bias) + addend."""
    a = torch.tensor([[3.0, 1.0]])
    b = torch.tensor([[100.0, 1.0]])                       # acc = 301
    bias = torch.tensor([0.5])
    add = torch.tensor([[2.0]]).bfloat16()
    got = X.expected_gemm(a, b, bias=bias, addend=add, out_dtype=torch.bfloat16)
    assert got.float().item() == 304.0                    # 303.5 -> 304 (bf16 ulp 2 at 256..512)
    got = X.expected_gemm(a, b, bias=bias, addend=add.float(), out_dtype=torch.float32)
    assert got.item() == 303.5


def test_compose_references():
    rng = np.random.default_rng(1)
    nb, fi, fo = 5, 3, 4
    w = X.int_tensor((nb, fi, fo), seed=1)
    comp = X.dyadic_weights((6, nb), seed=2)
    root = X.int_tensor((fi, fo), seed=3)
    live = [4, 1, 2]
    wn = X.expected_compose(w, comp, root, live, torch.float32, "agg")
    w64 = (comp.double()[live] @ w.double().view(nb, -1)).view(3, fi, fo)
    assert torch.equal(wn.double(), torch.cat([w64, root.double()[None]]).reshape(-1, fo))
    tf = X.expected_compose(w, comp, root, live, torch.float32, "tf")
    assert torch.equal(tf.double(), torch.cat([w64, root.double()[None]]).permute(1, 0, 2).reshape(fi, -1))
    dws = X.int_tensor((3, fi, fo), seed=5)
    dweight, dcomp = X.expected_compose_bwd(w, comp, dws, live)
    assert torch.equal(dweight.double(), torch.einsum("sb,sio->bio", comp.double()[live], dws.double()))
    want = torch.zeros(6, nb, dtype=torch.float64)
    want[live] = torch.einsum("sio,bio->sb", dws.double(), w.double())
    assert torch.equal(dcomp.double(), want)
    assert rng is not None


def test_pow2_graph_segments_are_powers_of_two():
    ei, et = X.pow2_graph(3000, 4, seed=1, hubs=[(3, 1024), (5, 256)], fanout_sources=3, fanout=500)
    src, dst, rel = ei[0].numpy(), ei[1].numpy(), et.numpy()
    seg = dst * 4 + rel
    counts = np.bincount(seg, minlength=3000 * 4)
    nz = counts[counts > 0]
    assert np.all(nz & (nz - 1) == 0)
    assert sorted(nz)[-3:] == [1024] * 3
    out_deg = np.bincount(src[rel == 3], minlength=3000)
    assert sorted(out_deg)[-3:] == [500] * 3
    assert src.max() < 3000 and dst.max() < 3000


def test_generators():
    t = X.int_tensor((1000,), torch.bfloat16, lo=-3, hi=3, nonzero=True, seed=2)
    v = set(t.float().tolist())
    assert v == {-3.0, -2.0, -1.0, 1.0, 2.0, 3.0}
    w = X.dyadic_weights(1000, seed=1)
    assert set(w.tolist()) == set(X.DYADIC)
    assert X.fraction_bits(w) == 2 and X.fraction_bits(t.float()) == 0
