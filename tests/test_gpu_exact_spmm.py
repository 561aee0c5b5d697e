"""The aggregation kernels (csrc/spmm.cu) bit for bit against ``exact_arith.expected_spmm`` on integer features and
dyadic weights, across their launch paths: every width class of ``launch_vec``, the four modes, strided inputs and
outputs, hub thresholds and row lengths at the threshold, group quanta, the band plan (rank key, id key, small
bands), every ``spmm_variant``, the overlapped hub path and the unroll switch.  The sum is exact whatever the
summation order, so one expected tensor holds for every path, and a reordering of the sums never changes it.

Where a case is meant to reach a path, the kernels it launches are read back from the profiler and asserted."""
import numpy as np
import pytest
import torch

import gmlm_b200 as G
from gmlm_b200 import _lib, synth
from gmlm_b200.graph import CSR, HUB_BAND_SHIFT

import exact_arith as X

pytestmark = pytest.mark.gpu

NO_HUBS = 1 << 30


def _launched(fn):
    """(result of fn(), names of the CUDA kernels it launched, spaces removed)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name.replace(" ", "") for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return out, names


def _assert_kernels(names, expect):
    for k in expect:
        assert any(k in n for n in names), f"{k} was not launched; launched: {sorted(names)}"


class _Tuning:
    """Process-wide tuning switches, restored on exit."""

    def __init__(self, **kv):
        self.kv, self.old = kv, {}

    def __enter__(self):
        for k, v in self.kv.items():
            self.old[k] = _lib.set_tuning(k, v)
        return self

    def __exit__(self, *exc):
        for k, v in self.old.items():
            _lib.set_tuning(k, v)


# ------------------------------------------------------------------------------ graphs (row lengths, columns)
def _graph(kind, thresh, seed):
    rng = np.random.default_rng(seed)
    if kind == "rmat":
        ei = synth.rmat_edges(3000, 40000, seed=seed).numpy()
        order = np.argsort(ei[1], kind="stable")
        return np.bincount(ei[1], minlength=3000), ei[0][order], 3000
    if kind == "star":                           # one row long enough for many chunks, then short rows
        lens = np.concatenate([[5000], rng.integers(0, 6, 300)])
    elif kind == "empty_runs":                   # long runs of empty rows between short and hub rows
        lens = np.zeros(6000, np.int64)
        at = rng.choice(6000, 120, replace=False)
        lens[at] = rng.integers(1, 40, 120)
        lens[at[:4]] = 700
    elif kind == "boundary":                     # rows of exactly hub_thresh and hub_thresh + 1 edges
        t = thresh if thresh < NO_HUBS else 256
        lens = np.array([t - 1, t, t + 1, 0, 2 * t, 2 * t + 1, 1, t + 1, 0, 0, t] * 7)
    elif kind == "n1":
        lens = np.array([7])
    elif kind == "nnz0":
        lens = np.zeros(10, np.int64)
    else:
        raise ValueError(kind)
    n_src = 1500
    return lens, rng.integers(0, n_src, int(lens.sum())), n_src


def _csr(lens, col, dev, w=None, thresh=256, quantum=0, bands="rank"):
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    c = CSR(rowptr=torch.tensor(rowptr, device=dev), col=torch.tensor(np.asarray(col, np.int32), device=dev),
            num_rows=len(lens), w=w, hub_thresh=thresh)
    c.plan_hubs()                                # the band plan with the rank key
    if bands == "id" and c.n_hub:
        c.plan_bands(HUB_BAND_SHIFT, rank=None)
    elif bands == "small" and c.n_hub:
        c.plan_bands(4, rank=c.col_rank())
    c.plan_groups(quantum)
    return c


# ------------------------------------------------------------------------------ the case matrix
F32, BF16 = torch.float32, torch.bfloat16
SUM, MEAN, W1, W2 = "sum", "mean", "w1", "w2"
MODE = {SUM: _lib.AGG_SUM, MEAN: _lib.AGG_MEAN, W1: _lib.AGG_WEIGHTED, W2: _lib.AGG_WEIGHTED}


def C(dtype, feat, mode, graph, thresh=256, quantum=0, heads=1, layout="plain", bands="rank", tuning=None,
      expect=(), hub=None, banded=None):
    """One case: ``expect`` = kernel names that must run; ``hub`` / ``banded``: the plan must (not) have hub rows /
    take the band plan (512-byte contiguous rows with a band plan)."""
    return dict(dtype=dtype, feat=feat, mode=mode, graph=graph, thresh=thresh, quantum=quantum, heads=heads,
                layout=layout, bands=bands, tuning=tuning or {}, expect=expect, hub=hub, banded=banded)


CASES = {
    # narrow kernels (<= 8 and <= 16 packs), sum / mean / 1-D weights, every quantum
    "f32_8p_sum_rmat_q0": C(F32, 32, SUM, "rmat", thresh=17, expect=("rows_narrow_kernel", "chunk_kernel"), hub=True),
    "f32_16p_mean_empty_q5": C(F32, 64, MEAN, "empty_runs", quantum=5, expect=("rows_narrow_kernel",), hub=True),
    "bf16_8p_w1_boundary17": C(BF16, 64, W1, "boundary", thresh=17, quantum=512, hub=True),
    "bf16_16p_mean_star_t1": C(BF16, 128, MEAN, "star", thresh=1, quantum=5, layout="out_view", hub=True),
    "f32_16p_w1_n1": C(F32, 64, W1, "n1", thresh=1, hub=True),
    "bf16_8p_sum_nnz0": C(BF16, 64, SUM, "nnz0", thresh=NO_HUBS, hub=False),
    "f32_8p_w1_nnz0": C(F32, 32, W1, "nnz0", thresh=17, hub=False),
    # the general kernel on narrow rows (variant 2, variant 0) and per-head weights (head slabs)
    "f32_8p_mean_rmat_v2": C(F32, 32, MEAN, "rmat", thresh=17, tuning=dict(spmm_variant=2),
                             expect=("rows_kernel", "chunk_kernel", "hub_final_kernel")),
    "bf16_16p_w1_empty_v0": C(BF16, 128, W1, "empty_runs", thresh=17, quantum=512, tuning=dict(spmm_variant=0),
                              expect=("rows_kernel",)),
    "f32_w2_h4_rmat": C(F32, 128, W2, "rmat", heads=4, thresh=17, quantum=5, expect=("rows_kernel",)),
    "bf16_w2_h2_boundary": C(BF16, 256, W2, "boundary", heads=2, thresh=256, layout="strided_x", hub=True),
    # one head slab above 128 packs: 520 fp32 features on 16-byte packs, 131 bf16 features on scalar packs
    "f32_w2_slab130p_star": C(F32, 1040, W2, "star", heads=2, thresh=17,
                              expect=("rows_kernel<float,4,8,32,1,1", "chunk_kernel<float,4,8,32,1,1")),
    "bf16_w2_slab131_rmat": C(BF16, 262, W2, "rmat", heads=2, thresh=256, quantum=5,
                              expect=("rows_kernel<__nv_bfloat16,1,8,32,1,1",)),
    # 512-byte rows: the band plan (rank key, id key, small bands), the bulk-copy chunk kernel, overlap, unroll 8
    "bf16_512B_mean_rmat_rank": C(BF16, 256, MEAN, "rmat", thresh=17, banded=True, expect=("chunk_kernel",)),
    "f32_512B_w1_star_id": C(F32, 128, W1, "star", thresh=17, quantum=5, bands="id", banded=True),
    "bf16_512B_w1_empty_small": C(BF16, 256, W1, "empty_runs", thresh=17, quantum=512, bands="small", banded=True),
    "f32_512B_mean_boundary_small": C(F32, 128, MEAN, "boundary", thresh=256, bands="small", banded=True),
    "bf16_512B_w1_rmat_v3": C(BF16, 256, W1, "rmat", thresh=17, bands="small", tuning=dict(spmm_variant=3),
                              banded=True, expect=("chunk_tma_kernel", "hub_final_kernel")),
    "f32_512B_mean_star_v4": C(F32, 128, MEAN, "star", thresh=17, tuning=dict(spmm_variant=4), banded=True,
                               expect=("chunk_tma_kernel",)),
    "bf16_512B_sum_boundary_v4_id": C(BF16, 256, SUM, "boundary", thresh=17, bands="id", quantum=5,
                                      tuning=dict(spmm_variant=4), banded=True, expect=("chunk_tma_kernel",)),
    "f32_512B_sum_rmat_v3_t1": C(F32, 128, SUM, "rmat", thresh=1, quantum=512, tuning=dict(spmm_variant=3),
                                 banded=True, expect=("chunk_tma_kernel",)),
    "bf16_512B_mean_empty_overlap": C(BF16, 256, MEAN, "empty_runs", thresh=17, tuning=dict(spmm_overlap=1),
                                      banded=True, expect=("rows_kernel", "chunk_kernel", "hub_final_kernel")),
    "f32_64p_w1_rmat_overlap": C(F32, 256, W1, "rmat", thresh=17, quantum=5, tuning=dict(spmm_overlap=1),
                                 layout="out_view", expect=("rows_kernel", "chunk_kernel")),
    "bf16_512B_w1_star_unroll8": C(BF16, 256, W1, "star", thresh=17, tuning=dict(spmm_unroll=8),
                                   expect=("rows_kernel<__nv_bfloat16,8,1,32,8,3",)),
    "f32_512B_sum_rmat_v0": C(F32, 128, SUM, "rmat", thresh=17, tuning=dict(spmm_variant=0), banded=True),
    "f32_512B_mean_rmat_nohub": C(F32, 128, MEAN, "rmat", thresh=NO_HUBS, quantum=5, hub=False),
    # a strided 512-byte input and a 512-byte column view as output take the CSR-order chunks
    "bf16_512B_mean_rmat_strided": C(BF16, 256, MEAN, "rmat", thresh=17, layout="strided_x", banded=False),
    "f32_512B_w1_star_outview": C(F32, 128, W1, "star", thresh=17, layout="out_view", tuning=dict(spmm_variant=3),
                                  banded=True),
    # wider rows: <= 64, <= 96 and > 96 packs
    "f32_64p_mean_star": C(F32, 256, MEAN, "star", thresh=17, quantum=512, hub=True),
    "bf16_64p_w1_rmat_strided": C(BF16, 512, W1, "rmat", thresh=256, layout="strided_x"),
    "f32_96p_w1_boundary": C(F32, 384, W1, "boundary", thresh=17, layout="out_view", hub=True),
    "bf16_96p_sum_empty": C(BF16, 768, SUM, "empty_runs", thresh=NO_HUBS, quantum=5, tuning=dict(spmm_variant=0)),
    "f32_wide_mean_rmat": C(F32, 520, MEAN, "rmat", thresh=17, layout="strided_x", tuning=dict(spmm_overlap=1)),
    "bf16_wide_w1_star": C(BF16, 1000, W1, "star", thresh=256, quantum=5, hub=True),
    # unaligned widths: scalar packs
    "f32_vec1_22_mean_rmat": C(F32, 22, MEAN, "rmat", thresh=17, expect=("rows_kernel<float,1,1,32",)),
    "f32_vec1_7_w1_empty": C(F32, 7, W1, "empty_runs", thresh=17, quantum=5, expect=("rows_narrow_kernel<float,1",)),
    "bf16_vec1_130_sum_boundary": C(BF16, 130, SUM, "boundary", thresh=17, layout="out_view", hub=True),
    "bf16_vec1_9_mean_n1": C(BF16, 9, MEAN, "n1", thresh=NO_HUBS, tuning=dict(spmm_variant=2)),
}


@pytest.mark.parametrize("name", list(CASES))
def test_spmm_exact(cuda_dev, name):
    c = CASES[name]
    dtype, feat, mode, heads = c["dtype"], c["feat"], MODE[c["mode"]], c["heads"]
    seed = sum(map(ord, name))
    lens, col, n_src = _graph(c["graph"], c["thresh"], seed)
    nnz = int(np.sum(lens))
    w = None
    if c["mode"] == W1:
        w = X.dyadic_weights(nnz, seed=seed + 1, device=cuda_dev)
    elif c["mode"] == W2:
        w = X.dyadic_weights((nnz, heads), seed=seed + 1, device=cuda_dev)
    csr = _csr(lens, col, cuda_dev, w=w, thresh=c["thresh"], quantum=c["quantum"], bands=c["bands"])
    if c["hub"] is not None:
        assert (csr.n_hub > 0) == c["hub"]
    if c["graph"] == "boundary":                        # rows of exactly thresh edges stay off the hub path
        t = c["thresh"]
        assert csr.n_hub == (int(np.sum(lens > t)) if t < NO_HUBS else 0)
    esz = 4 if dtype == F32 else 2
    if c["layout"] == "strided_x":
        x = X.int_tensor((n_src, feat + 24), dtype, seed=seed + 2, device=cuda_dev)[:, 8:8 + feat]
    else:
        x = X.int_tensor((n_src, feat), dtype, seed=seed + 2, device=cuda_dev)
    if c["banded"] is not None:
        assert csr.n_hub > 0 and feat * esz == 512
        takes_bands = csr.band_plan is not None and x.is_contiguous() and c["mode"] != W2
        assert takes_bands == c["banded"]
        if c["mode"] == W1 and c["banded"]:
            assert csr.hub_w is not None
    if c["bands"] == "small":
        assert csr.n_band_chunks > csr.n_chunks          # band boundaries cut chunks
    want = X.expected_csr_spmm(x, csr, mode)

    buf = None
    if c["layout"] == "out_view":
        off = 16 if feat % (16 // esz) == 0 else 3       # keeps an aligned view aligned (16-byte offset and pitch)
        buf = torch.full((csr.num_rows, feat + 2 * off), float("nan"), dtype=dtype, device=cuda_dev)

    def run():
        if buf is not None:
            return G.spmm(x, csr, mode, out=buf[:, off:off + feat])
        return G.spmm(x, csr, mode)

    with _Tuning(**c["tuning"]):
        if c["expect"]:
            got, names = _launched(run)
            _assert_kernels(names, c["expect"])
        else:
            got = run()
        again = run()
    assert got.dtype == dtype and got.shape == (csr.num_rows, feat)
    assert torch.equal(got.cpu(), want), name
    assert torch.equal(again, got)
    if buf is not None:
        assert torch.isnan(buf[:, :off]).all() and torch.isnan(buf[:, off + feat:]).all()


# ------------------------------------------------------------------------------ the layer paths
@pytest.fixture(scope="module")
def pow2_big(cuda_dev):
    """160k nodes, every (dst, rel) segment a power of two long: hub segments of 512 and 4096 edges that gather from
    more rows than two bands of the hub plan hold, and sources that feed 600 segments each (hub rows of the
    transposed CSR).  The 1/|segment| weights are dyadic, so the backward is exact too."""
    ei, et = X.pow2_graph(160_000, 4, seed=5, p_empty=0.7, hubs=[(24, 4096), (40, 512)], fanout_sources=8,
                          fanout=600)
    g = G.RelGraph.build(ei.to(cuda_dev), et.to(cuda_dev), 160_000, 4)
    for csr in (g.fwd, g.bwd):
        assert csr.n_hub > 0 and csr.band_plan is not None
    rank = g.fwd.col_rank()
    assert (int(rank[g.fwd.hub_col.long()].max()) >> HUB_BAND_SHIFT) + 1 >= 3   # three bands of source rows
    return g


@pytest.mark.parametrize("dtype,feat", [(F32, 128), (BF16, 256), (BF16, 64)])
def test_rgcn_aggregate_exact(pow2_big, dtype, feat):
    """Forward mean and backward 1/|segment|-weighted gather through the autograd op, bit for bit."""
    g = pow2_big
    n, S = g.num_nodes, g.num_slots
    x = X.int_tensor((n, feat), dtype, seed=feat, device="cuda").requires_grad_(True)
    h = G.rgcn_aggregate(x, g)
    assert torch.equal(h.detach().view(n * S, feat).cpu(), X.expected_csr_spmm(x.detach(), g.fwd, _lib.AGG_MEAN))
    gh = X.int_tensor((n * S, feat), dtype, seed=feat + 1, device="cuda")
    h.backward(gh.view_as(h))
    if feat * x.element_size() == 512:
        assert g.bwd.hub_w is not None                  # the weighted band path
    assert torch.equal(x.grad.cpu(), X.expected_csr_spmm(gh, g.bwd, _lib.AGG_WEIGHTED))


@pytest.mark.parametrize("dtype,fo", [(F32, 128), (BF16, 256)])
@pytest.mark.parametrize("plan", ["dst", "seg"])
def test_transform_first_and_segment_compact_plans_exact(pow2_big, dtype, fo, plan):
    """The CSRs of the transform-first (``dst_plan``) and segment-compact (``seg_plan``) formulations at 512-byte
    rows: the weighted band path with ``hub_w`` in both directions of the transform-first plan."""
    g = pow2_big
    if plan == "dst":
        f, b = g.dst_plan()
        fwd_mode = _lib.AGG_WEIGHTED
        n_in = g.num_src * (g.num_slots + 1)
    else:
        p = g.seg_plan()
        f, b = p.fwd, p.bwd
        fwd_mode = _lib.AGG_MEAN
        n_in = g.num_src
    for csr, mode, rows_in in ((f, fwd_mode, n_in), (b, _lib.AGG_WEIGHTED, f.num_rows)):
        assert csr.n_hub > 0 and csr.band_plan is not None
        if mode == _lib.AGG_WEIGHTED:
            assert csr.hub_w is not None
        x = X.int_tensor((rows_in, fo), dtype, seed=rows_in % 1000, device="cuda")
        got = G.spmm(x, csr, mode)
        assert torch.equal(got.cpu(), X.expected_csr_spmm(x, csr, mode)), (plan, mode)
