"""The band-ordered hub plan (``CSR.plan_bands``, csrc/graph_build.cu) against a numpy restatement, integer-exact,
and the aggregation on 512-byte rows that runs it (csrc/spmm.cu) against fp64 on graphs whose hub rows span several
bands of source rows."""
import numpy as np
import pytest
import torch

import gmlm_b200 as G
from gmlm_b200 import _lib, synth
from gmlm_b200.graph import HUB_BAND_MIN_RUN, HUB_BAND_SHIFT

from conftest import rel_err

pytestmark = pytest.mark.gpu


def plan_ref(rowptr, col, w, thresh, shift, min_run):
    """(hub_col, hub_w, band_chunk_ptr, cut, chunk_order) as include/gmlm_b200.h defines them."""
    lens = np.diff(rowptr)
    hub_rows = np.nonzero(lens > thresh)[0]
    hub_col, hub_w, chunk_ptr, cut = [], [], [0], []
    pos = 0
    for r in hub_rows:
        a, b = rowptr[r], rowptr[r + 1]
        order = np.argsort(col[a:b], kind="stable")
        c = col[a:b][order]
        hub_col.append(c)
        if w is not None:
            hub_w.append(w[a:b][order])
        band = c >> shift
        bounds = [int(p) for p in np.nonzero(band[1:] != band[:-1])[0] + 1]   # band boundaries inside the row
        last = 0
        kept = []
        for p in bounds:
            if p - last >= min_run and len(c) - p >= min_run:
                kept.append(p)
                last = p
        starts = []
        for lo, hi in zip([0] + kept, kept + [len(c)]):
            starts.extend(range(lo, hi, thresh))
        cut.extend(pos + s for s in starts)
        chunk_ptr.append(chunk_ptr[-1] + len(starts))
        pos += len(c)
    cut.append(pos)
    hub_col = np.concatenate(hub_col) if hub_col else np.zeros(0, np.int64)
    cut = np.asarray(cut, np.int64)
    first_band = hub_col[cut[:-1]] >> shift
    order = np.argsort(first_band, kind="stable")
    return (hub_col, np.concatenate(hub_w) if hub_w else None, np.asarray(chunk_ptr), cut, order)


def _graph(n, e, seed, thresh):
    ei = synth.rmat_edges(n, e, seed=seed).cuda()
    et = G.edge_type_from_degree(ei, n)
    return G.RelGraph.build(ei, et, n, 5, hub_thresh=thresh)


def _check_plan(csr, shift):
    rp = csr.rowptr.cpu().numpy().astype(np.int64)
    col = csr.col.cpu().numpy().astype(np.int64)
    w = csr.w.cpu().numpy() if csr.w is not None else None
    hub_col, hub_w, chunk_ptr, cut, order = plan_ref(rp, col, w, csr.hub_thresh, shift, HUB_BAND_MIN_RUN)
    nh, nb = csr.n_hub, csr.n_band_chunks
    bp = csr.band_plan.cpu().numpy().astype(np.int64)
    assert bp.size == nh + 2 + 2 * nb
    np.testing.assert_array_equal(csr.hub_col.cpu().numpy(), hub_col)
    if w is not None:
        np.testing.assert_array_equal(csr.hub_w.cpu().numpy(), hub_w)      # bit-exact: a permutation of w
    else:
        assert csr.hub_w is None
    np.testing.assert_array_equal(bp[:nh + 1], chunk_ptr)                     # partial slots grouped by row
    np.testing.assert_array_equal(bp[nh + 1:nh + 2 + nb], cut)
    np.testing.assert_array_equal(bp[nh + 2 + nb:], order)
    # every chunk: at most hub_thresh edges, inside one hub row
    lens = np.diff(cut)
    assert lens.min() >= 1 and lens.max() <= csr.hub_thresh
    return nb


@pytest.mark.parametrize("shift", [6, 10, HUB_BAND_SHIFT])
def test_band_plan_matches_numpy(cuda_dev, shift):
    g = _graph(20_000, 400_000, seed=3, thresh=64)
    for csr in (g.fwd, g.bwd):
        assert csr.n_hub > 0
        csr.plan_bands(shift)
        nb = _check_plan(csr, shift)
        if shift <= 10:
            assert nb > csr.n_chunks            # band boundaries did cut chunks
        csr.plan_bands()


def test_band_plan_min_run_rule(cuda_dev):
    """Hand-made rows: boundaries that leave a piece under HUB_BAND_MIN_RUN edges are not cuts."""
    shift = 4
    m = HUB_BAND_MIN_RUN
    rows = [
        [0] * 40 + [16] * 40 + [32] * 40,              # two kept cuts
        [0] * 5 + [16] * 100 + [32] * 5,               # short first and last pieces: no cut, hub_thresh tiles
        [0] * 40 + [16] * 3 + [32] * 60,               # the boundary at 40 is kept, the one at 43 is not
        list(range(0, 16 * 300, 16)),                  # a new band every edge: cuts every min_run edges, the
                                                       # last piece keeps >= min_run (44 edges)
    ]
    rng = np.random.default_rng(0)
    rowptr = np.zeros(len(rows) + 1, np.int64)
    rowptr[1:] = np.cumsum([len(r) for r in rows])
    col = np.concatenate([rng.permutation(np.asarray(r)) for r in rows])
    csr = G.graph.CSR(rowptr=torch.tensor(rowptr, dtype=torch.int32, device=cuda_dev),
                      col=torch.tensor(col, dtype=torch.int32, device=cuda_dev), num_rows=len(rows), hub_thresh=64)
    csr.plan_hubs()
    assert csr.n_hub == len(rows)
    csr.plan_bands(shift)
    _check_plan(csr, shift)
    bp = csr.band_plan.cpu().numpy()
    cut = bp[len(rows) + 1:len(rows) + 2 + csr.n_band_chunks]
    assert list(cut[:7]) == [0, 40, 80, 120, 184, 230, 270]
    assert list(cut[7:]) == [333 + m * k for k in range(9)] + [633]


def _ref(x64, csr, mode):
    rp = csr.rowptr.long()
    lens = rp[1:] - rp[:-1]
    rows = torch.repeat_interleave(torch.arange(csr.num_rows, device=rp.device), lens)
    col = csr.col.long()
    out = torch.zeros(csr.num_rows, x64.size(1), dtype=torch.float64, device=x64.device)
    for a in range(0, col.numel(), 1 << 18):
        b = min(col.numel(), a + (1 << 18))
        v = x64[col[a:b]]
        if mode == _lib.AGG_WEIGHTED:
            v = v * csr.w[a:b].double()[:, None]
        out.index_add_(0, rows[a:b], v)
    if mode == _lib.AGG_MEAN:
        out /= lens.clamp(min=1).double()[:, None]
    return out


def _without_bands(csr):
    c = G.graph.CSR(**{k: getattr(csr, k) for k in csr.__dataclass_fields__})
    c.hub_col = c.hub_w = c.band_plan = None
    return c


@pytest.fixture(scope="module")
def multi_band_graph(cuda_dev):
    """300k nodes: hub rows gather from more than 2^HUB_BAND_SHIFT source rows, i.e. from several bands; a hub
    threshold of 32 puts most edges on the hub path."""
    g = _graph(300_000, 3_000_000, seed=11, thresh=32)
    bands = (g.fwd.hub_col.max().item() >> HUB_BAND_SHIFT) + 1
    assert bands >= 3
    return g


@pytest.mark.parametrize("dtype,feat", [(torch.bfloat16, 256), (torch.float32, 128)])
def test_banded_aggregation_fp64(multi_band_graph, dtype, feat):
    g = multi_band_graph
    n, S = g.num_nodes, g.num_slots
    x = synth.make_features(n, feat, device="cuda", seed=1, dtype=dtype)
    gh = synth.make_features(n * S, feat, device="cuda", seed=2, dtype=dtype)
    tol = 2e-2 if dtype == torch.bfloat16 else 1e-5
    for csr, inp, mode in ((g.fwd, x, _lib.AGG_MEAN), (g.bwd, gh, _lib.AGG_WEIGHTED)):
        hub_edges = int(csr.hub_col.numel())
        assert hub_edges > csr.nnz // 4
        out = G.spmm(inp, csr, mode)
        ref = _ref(inp.double(), csr, mode)
        assert rel_err(out, ref) < tol
        assert torch.equal(out, G.spmm(inp, csr, mode))                 # run to run: bit-identical
        buf = torch.empty_like(out)
        assert torch.equal(out, G.spmm(inp, csr, mode, out=buf))       # the out= path runs the same plan
        # the hub rows took the band plan (source order), the other rows are the rows kernel's, bit for bit
        plain = G.spmm(inp, _without_bands(csr), mode)
        hub = torch.zeros(csr.num_rows, dtype=torch.bool, device=out.device)
        hub[csr.hub_row.long()] = True
        assert torch.equal(out[~hub], plain[~hub])
        assert not torch.equal(out[hub], plain[hub])
        assert rel_err(out[hub], plain[hub]) < tol


def test_rgcn_aggregate_autograd_uses_bands(multi_band_graph):
    g = multi_band_graph
    n, S = g.num_nodes, g.num_slots
    x = synth.make_features(n, 256, device="cuda", seed=3, dtype=torch.bfloat16).requires_grad_(True)
    h = G.rgcn_aggregate(x, g)
    assert torch.equal(h.view(n * S, 256), G.spmm(x.detach(), g.fwd, _lib.AGG_MEAN))
    gh = synth.make_features(n * S, 256, device="cuda", seed=4, dtype=torch.bfloat16)
    h.backward(gh.view_as(h))
    assert torch.equal(x.grad, G.spmm(gh, g.bwd, _lib.AGG_WEIGHTED))


@pytest.mark.parametrize("case", ["strided_512B", "fp32_1KB"])
def test_other_rows_keep_the_csr_order_chunks(multi_band_graph, case):
    """A 512-byte view with ldx > feat and 1 KB rows take the CSR-order hub chunks: bit-identical to a CSR
    without a band plan, and still right against fp64."""
    g = multi_band_graph
    n = g.num_nodes
    if case == "strided_512B":
        x = synth.make_features(n, 320, device="cuda", seed=5, dtype=torch.bfloat16)[:, :256]
        tol = 2e-2
    else:
        x = synth.make_features(n, 256, device="cuda", seed=5, dtype=torch.float32)
        tol = 1e-5
    out = G.spmm(x, g.fwd, _lib.AGG_MEAN)
    assert torch.equal(out, G.spmm(x, _without_bands(g.fwd), _lib.AGG_MEAN))
    assert rel_err(out, _ref(x.double(), g.fwd, _lib.AGG_MEAN)) < tol
