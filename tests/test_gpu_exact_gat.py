"""The fused GAT kernels (gmlm_b200/csrc/gat_fused.cu) on binary attention: every score is either the row's maximum
or at least 200 below it, where exp underflows to exactly 0 in fp32, so out[i,h] is the mean of the integer z[j,h]
over the edges that share the row's maximum score (2x the sum over the kept ones with dropout 0.5).  The sums are
exact; the only rounding left is the division by the count, so every element is gated at 1 ulp of the output type.
Covers 1-32 heads on the vectorised, scalar-pack and head-group instances, hub rows whose chunks are all hidden (the
(m, l) merge of gat_final_kernel), the backward (dz exact on power-of-two counts, the score gradients against fp64
with a bound built from the sums of |terms|) and the self-loop fill with fill_value="mean"."""
import numpy as np
import pytest
import torch

from gmlm_b200.attn import LoopGraph, gat_aggregate, gat_dropout_mask, gat_edge_scores

import exact_arith as X
from test_gpu_exact_spmm import _assert_kernels, _launched

pytestmark = pytest.mark.gpu

HIDE = -1000.0
F32, BF16 = torch.float32, torch.bfloat16
N, N_HUB, HUB_LEN, BEACONS = 3000, 6, 2500, 10


@pytest.fixture(scope="module")
def gat_graph():
    """Uniform edges with self-loops and duplicates, plus hub rows of 2500 in-edges from the upper half of the nodes
    (whose a_src hides them below) and three from the first BEACONS nodes, hub_thresh = 32: most chunks of a hub
    row are all hidden."""
    rng = np.random.default_rng(5)
    src = [rng.integers(0, N, 30000)]
    dst = [rng.integers(0, N, 30000)]
    src.append(np.arange(0, N, 7))
    dst.append(np.arange(0, N, 7))
    for h in range(N_HUB):
        src.append(np.concatenate([rng.integers(N // 2, N, HUB_LEN), rng.integers(0, BEACONS, 3 if h else 0)]))
        dst.append(np.full(src[-1].size, 100 + h))
    ei = torch.tensor(np.stack([np.concatenate(src), np.concatenate(dst)]), device="cuda")
    graph = LoopGraph.build(ei, N, hub_thresh=32)
    assert graph.fwd.n_hub >= N_HUB
    return ei, graph


def _csr_np(graph):
    rowptr = graph.fwd.rowptr.cpu().numpy().astype(np.int64)
    col = graph.fwd.col.cpu().numpy().astype(np.int64)[:rowptr[-1]]
    return rowptr, col, np.repeat(np.arange(rowptr.size - 1), np.diff(rowptr))


def _visible(raw32, dst, n, slope=np.float32(0.2)):
    """Edges whose score equals their row's maximum (per head)."""
    s = np.where(raw32 > 0, raw32, raw32 * slope)
    mx = np.full((n, s.shape[1]), -np.inf, np.float32)
    np.maximum.at(mx, dst, s)
    return s == mx[dst]


def _expected_out(z, col, dst, vis, w, n, heads):
    """(sum over edges of w * z[col] in fp64, visible count) per row and head."""
    c = z.size(1) // heads
    z64 = z.double().cpu().view(-1, heads, c)[torch.from_numpy(col)]
    acc = torch.zeros(n, heads, c, dtype=torch.float64).index_add_(
        0, torch.from_numpy(dst), torch.from_numpy(w)[:, :, None] * z64)
    cnt = torch.zeros(n, heads, dtype=torch.float64).index_add_(0, torch.from_numpy(dst), torch.from_numpy(vis * 1.0))
    return acc, cnt


def _within_one_ulp(got, want64, dtype, what):
    """got within one step of the output type of the correctly rounded want (the kernels' scale by 1 / count
    rounds twice)."""
    want = X.round_to(want64.float().numpy(), dtype).double() if dtype != F32 else want64.float().double()
    got = got.double().cpu()
    mag = torch.maximum(want.abs(), got.abs()).clamp(min=2.0 ** -100)
    ulp = torch.pow(2.0, torch.floor(torch.log2(mag)) - (23 if dtype == F32 else 7))
    bad = (got - want).abs() > ulp
    if bad.any():
        i = tuple(bad.nonzero()[0].tolist())
        raise AssertionError(f"{what}: {int(bad.sum())} elements off by more than 1 ulp; at {i}: got "
                             f"{got[i].item()}, want {want64[i].item()}")


def _keep(graph, heads, p, seed):
    if p == 0:
        return np.ones((graph.fwd.nnz, heads)), 1.0
    return gat_dropout_mask(seed, graph.fwd.nnz, heads, p, "cuda").cpu().numpy() * 1.0, 1.0 / (1.0 - p)


# (dtype, heads, head_dim, dropout, instance that must run -- the chunk kernel of the rows kernel's dispatch):
# 16-byte packs at CH 1/2/4/8, scalar packs, head groups
FWD = [(F32, 1, 64, 0.0, "gat_chunk_kernel<float,4,1,false"), (F32, 4, 32, 0.5, "gat_chunk_kernel<float,4,1,false"),
       (F32, 32, 8, 0.0, "gat_chunk_kernel<float,4,2,false"), (F32, 16, 64, 0.5, "gat_chunk_kernel<float,4,8,false"),
       (F32, 32, 64, 0.0, "gat_chunk_kernel<float,4,8,true"), (F32, 3, 7, 0.5, "gat_chunk_kernel<float,1,1,false"),
       (F32, 32, 9, 0.5, "gat_chunk_kernel<float,1,8,true"), (BF16, 2, 64, 0.5, "gat_chunk_kernel<__nv_bfloat16,8,1,false"),
       (BF16, 8, 128, 0.0, "gat_chunk_kernel<__nv_bfloat16,8,4,false"),
       (BF16, 16, 128, 0.5, "gat_chunk_kernel<__nv_bfloat16,8,4,true"),
       (BF16, 5, 11, 0.0, "gat_chunk_kernel<__nv_bfloat16,1,4,false"),
       (BF16, 32, 10, 0.5, "gat_chunk_kernel<__nv_bfloat16,1,8,true")]


@pytest.mark.parametrize("dtype,heads,c,p,kernel", FWD, ids=[f"{str(f[0])[6:]}-h{f[1]}-c{f[2]}-p{f[3]}" for f in FWD])
def test_gat_forward_binary_attention_within_one_ulp(cuda_dev, gat_graph, dtype, heads, c, p, kernel):
    """Scores from a_src alone (0 or -1000 per source and head, a_dst = 1): the row mean over the sources that
    share the row's maximum, self-loop included; with dropout, 2x the sum over the kept ones by the same count."""
    _, graph = gat_graph
    rowptr, col, dst = _csr_np(graph)
    rng = np.random.default_rng(heads * 100 + c)
    a_src = np.where(rng.random((N, heads)) < 0.5, 0.0, HIDE).astype(np.float32)
    a_src[N // 2:] = HIDE                                   # the hub rows' bulk: hidden in every head
    a_dst = np.ones((N, heads), np.float32)
    z = X.int_tensor((N, heads * c), dtype, seed=heads + c, device="cuda")
    seed = 1234 + heads
    keep, scale = _keep(graph, heads, p, seed)
    vis = _visible(a_src[col] + a_dst[dst], dst, N)
    # the merge case is real: a hub row with a visible edge in one chunk and chunks with none
    beg, end = graph.fwd.chunk_beg.cpu().numpy(), graph.fwd.chunk_end.cpu().numpy()
    hidden_chunk = np.array([not vis[b:e, 0].any() for b, e in zip(beg, end)])
    assert hidden_chunk.sum() > 10 and (~hidden_chunk).any()
    out, names = _launched(lambda: gat_aggregate(z, torch.from_numpy(a_src).cuda(), torch.from_numpy(a_dst).cuda(),
                                                 graph, 0.2, p, seed))
    _assert_kernels(names, (kernel, "gat_chunk_kernel", "gat_final_kernel"))
    acc, cnt = _expected_out(z, col, dst, vis, vis * keep * scale, N, heads)
    _within_one_ulp(out, (acc / cnt[:, :, None]).view(N, heads * c), dtype, "out")


def _pow2_visible(rowptr, heads, rng):
    """Per row and head, a random subset of a power-of-two size (at least 1) of the row's edges."""
    vis = np.zeros((rowptr[-1], heads), bool)
    for r in range(rowptr.size - 1):
        b, e = rowptr[r], rowptr[r + 1]
        for h in range(heads):
            k = 1 << int(rng.integers(0, int(np.log2(e - b)) + 1))
            vis[b + rng.choice(e - b, k, replace=False), h] = True
    return vis


BWD = [(F32, 4, 32, 0.5), (BF16, 8, 128, 0.0), (F32, 32, 64, 0.5), (BF16, 32, 10, 0.5), (F32, 1, 5, 0.0)]


@pytest.mark.parametrize("dtype,heads,c,p", BWD, ids=[f"{str(f[0])[6:]}-h{f[1]}-c{f[2]}-p{f[3]}" for f in BWD])
def test_gat_backward_binary_attention(cuda_dev, gat_graph, dtype, heads, c, p):
    """Scores from a_edge alone (0 or -1000 per edge and head), power-of-two visible counts: the alphas are dyadic,
    so out and dz (a weighted spmm of g with per-head weights over the transposed CSR) are exact; d_score, da_src
    and da_dst against fp64 within a bound built from the sums of |terms|."""
    _, graph = gat_graph
    rowptr, col, dst = _csr_np(graph)
    nnz = rowptr[-1]
    rng = np.random.default_rng(heads * 10 + c)
    vis = _pow2_visible(rowptr, heads, rng)
    a_edge = np.where(vis, 0.0, HIDE).astype(np.float32)
    z = X.int_tensor((N, heads * c), dtype, seed=c, device="cuda").requires_grad_(True)
    gout = X.int_tensor((N, heads * c), dtype, seed=c + 1, device="cuda")
    a_src = torch.zeros(N, heads, device="cuda", requires_grad=True)
    a_dst = torch.ones(N, heads, device="cuda", requires_grad=True)
    seed = 99 + heads
    keep, scale = _keep(graph, heads, p, seed)
    out = gat_aggregate(z, a_src, a_dst, graph, 0.2, p, seed, a_edge=torch.from_numpy(a_edge).cuda())
    out.backward(gout)
    acc, cnt = _expected_out(z.detach(), col, dst, vis, vis * keep * scale, N, heads)
    assert np.all(cnt.numpy() == 2.0 ** np.round(np.log2(cnt.numpy())))
    out64 = (acc / cnt[:, :, None]).view(N, heads * c)
    assert torch.equal(out.cpu(), X.round_to(out64.float().numpy(), dtype))
    # dz: sum over the out-edges of alpha_eff * g[dst], alpha_eff = keep * scale / count
    alpha = vis / cnt.numpy()[dst]
    order = np.argsort(col, kind="stable")
    rp_t = np.concatenate([[0], np.cumsum(np.bincount(col, minlength=N))])
    w_t = torch.from_numpy((alpha * keep * scale)[order])
    assert torch.equal(z.grad.cpu(), X.expected_spmm(gout.cpu(), rp_t, dst[order], X.AGG_WEIGHTED, w_t))
    # the score gradients: d_score = alpha (keep scale <g_i, z_j> - <g_i, out_i>) on visible edges (raw = 1 > 0),
    # 0 on hidden ones; a_edge's gradient is d_score, a_dst's the row sum, a_src's the column sum
    g64 = gout.double().cpu().view(N, heads, c)
    z64 = z.detach().double().cpu().view(N, heads, c)
    o64 = out.detach().double().cpu().view(N, heads, c)
    dot = (g64[dst] * z64[col]).sum(-1).numpy()
    t = (g64 * o64).sum(-1).numpy()[dst]
    ks = keep * scale
    d_score = alpha * (ks * dot - t)
    bound = 2.0 ** -20 * alpha * (ks * (g64[dst].abs() * z64[col].abs()).sum(-1).numpy()
                                  + (g64.abs() * o64.abs()).sum(-1).numpy()[dst])
    da_dst = np.zeros((N, heads))
    np.add.at(da_dst, dst, d_score)
    b_dst = np.zeros((N, heads))
    np.add.at(b_dst, dst, bound + 2.0 ** -22 * np.abs(d_score) * np.diff(rowptr)[dst, None])
    da_src = np.zeros((N, heads))
    np.add.at(da_src, col, d_score)
    b_src = np.zeros((N, heads))
    np.add.at(b_src, col, bound + 2.0 ** -22 * np.abs(d_score) * np.bincount(col, minlength=N)[col, None])
    for what, got, want, b in (("da_dst", a_dst.grad, da_dst, b_dst), ("da_src", a_src.grad, da_src, b_src)):
        err = np.abs(got.cpu().double().numpy() - want)
        assert np.all(err <= b), f"{what}: worst excess {np.max(err - b)}"
    assert nnz == graph.fwd.nnz


@pytest.mark.parametrize("heads", [1, 3, 32])
def test_gat_loop_fill_mean_within_one_ulp(cuda_dev, gat_graph, heads):
    """gat_edge_scores (fill_value="mean"): the kept edges' integer scores unchanged in forward-CSR order, each
    node's loop the mean over its kept in-edges (0 without), within 1 ulp of fp32."""
    ei, graph = gat_graph
    alpha = X.int_tensor((ei.size(1), heads), F32, seed=heads, device="cuda")
    got = gat_edge_scores(alpha, graph).cpu()
    ei_c, al = ei.cpu(), alpha.double().cpu()
    kept = ei_c[0] != ei_c[1]
    s = torch.zeros(N, heads, dtype=torch.float64).index_add_(0, ei_c[1][kept], al[kept])
    cnt = torch.zeros(N, dtype=torch.float64).index_add_(0, ei_c[1][kept], torch.ones(int(kept.sum()),
                                                                                   dtype=torch.float64))
    csr_src = graph.csr_src.cpu().long()
    want = torch.empty(graph.fwd.nnz, heads, dtype=torch.float64)
    want[csr_src >= 0] = al[csr_src[csr_src >= 0]]
    want[graph.loop_csr.cpu().long()] = s / cnt.clamp(min=1)[:, None]
    assert torch.equal(got[csr_src >= 0].double(), want[csr_src >= 0])
    _within_one_ulp(got, want, F32, "loop fill")
