"""N3 on the GPU: the reference's edge dropout (``augment_graph``, main.py:832-837) fused into the degree
histogram, the edge typing and the CSR build as a keep MASK must give, array for array, the graph built from the
filtered ``edge_index`` -- and the saved / reloaded CSR must aggregate identically."""
import numpy as np
import pytest
import torch

import gmlm_b200 as G
from gmlm_b200 import _lib, synth
from gmlm_b200.ingest import build_dropped_graph, edge_dropout_mask, load_rel_graph, save_rel_graph

import exact_arith as X

pytestmark = pytest.mark.gpu


def _same_csr(a, b):
    for k in ("rowptr", "col", "perm", "w", "grp_row", "hub_row", "hub_chunk_ptr", "chunk_beg", "chunk_end", "hub_col",
              "hub_w", "band_plan"):
        x, y = getattr(a, k), getattr(b, k)
        assert (x is None) == (y is None), k
        if x is not None and k != "perm":
            assert torch.equal(x, y), k
    assert (a.num_rows, a.n_hub, a.n_chunks, a.n_groups) == (b.num_rows, b.n_hub, b.n_chunks, b.n_groups)


@pytest.mark.parametrize("n,e,p", [(500, 8000, 0.1), (3000, 60000, 0.5), (40, 300, 0.9), (10, 50, 0.0)])
def test_fused_edge_dropout_equals_filtered_build(cuda_dev, n, e, p):
    ei = synth.rmat_edges(n, e, seed=n)
    keep = edge_dropout_mask(e, p, generator=torch.Generator().manual_seed(3))
    ei_d = ei.to(cuda_dev)
    fused = build_dropped_graph(ei_d, keep, n)
    ei_f = ei[:, keep].to(cuda_dev)                                         # what the reference materialises
    et_f = G.edge_type_from_degree(ei_f, n)
    want = G.RelGraph.build(ei_f, et_f, n, 5)
    assert fused.num_edges == want.num_edges == int(keep.sum()) and fused.live_rels == want.live_rels
    _same_csr(fused.fwd, want.fwd)
    _same_csr(fused.bwd, want.bwd)
    # perm refers to positions in the UNFILTERED edge list: map through the kept positions
    kept_pos = torch.nonzero(keep).squeeze(1).to(cuda_dev)
    assert torch.equal(fused.fwd.perm.long(), kept_pos[want.fwd.perm.long()])
    x = torch.randn(n, 32, device=cuda_dev)
    assert torch.equal(G.rgcn_aggregate(x, fused), G.rgcn_aggregate(x, want))


def test_rel_graph_file_round_trip(cuda_dev, tmp_path):
    n, e = 2000, 40000
    ei = synth.rmat_edges(n, e, seed=2).to(cuda_dev)
    g = G.RelGraph.build(ei, G.edge_type_from_degree(ei, n), n, 5, hub_thresh=64)
    path = str(tmp_path / "graph.pt")
    save_rel_graph(g, path)
    g2 = load_rel_graph(path, cuda_dev)
    _same_csr(g.fwd, g2.fwd)
    _same_csr(g.bwd, g2.bwd)
    x = torch.randn(n, 64, device=cuda_dev, requires_grad=True)
    h1, h2 = G.rgcn_aggregate(x, g), G.rgcn_aggregate(x, g2)
    assert torch.equal(h1, h2)
    gh = torch.randn_like(h1)
    assert torch.equal(torch.autograd.grad((h1 * gh).sum(), x)[0], torch.autograd.grad((h2 * gh).sum(), x)[0])
    with pytest.raises(G.GmlmError):
        load_rel_graph(path, "cpu")


def test_dropout_built_and_reloaded_band_plans_aggregate_exactly(cuda_dev, tmp_path):
    """512-byte integer rows through the band plans of a graph built with a keep mask and of its saved / reloaded
    copy: forward mean and backward 1/|segment|-weighted gather bit for bit against the exact reference.  The mask
    drops whole (dst, rel) segments or the second half of one, so every kept segment stays a power of two long and
    the backward weights stay dyadic."""
    n, R = 5000, 4
    ei, et = X.pow2_graph(n, R, seed=9, hubs=[(6, 1024), (10, 128)], fanout_sources=4, fanout=200)
    seg = (ei[1] * R + et).numpy()
    order = np.argsort(seg, kind="stable")
    lens = np.bincount(seg, minlength=n * R)
    start = np.concatenate([[0], np.cumsum(lens)])[:-1]
    rank = np.empty(seg.size, np.int64)
    rank[order] = np.arange(seg.size) - start[seg[order]]
    action = np.random.default_rng(1).choice(3, size=n * R, p=[0.6, 0.2, 0.2])[seg]   # keep / drop / halve
    keep = torch.from_numpy((action == 0) | ((action == 2) & (rank < lens[seg] // 2)))
    ei_d, et_d = ei.to(cuda_dev), et.to(cuda_dev)
    g = G.RelGraph.build(ei_d, et_d, n, R, hub_thresh=64, keep_mask=keep.to(cuda_dev))
    want = G.RelGraph.build(ei_d[:, keep.to(cuda_dev)], et_d[keep.to(cuda_dev)], n, R, hub_thresh=64)
    _same_csr(g.fwd, want.fwd)
    _same_csr(g.bwd, want.bwd)
    path = str(tmp_path / "graph.pt")
    save_rel_graph(g, path)
    g2 = load_rel_graph(path, cuda_dev)
    _same_csr(g.fwd, g2.fwd)
    _same_csr(g.bwd, g2.bwd)
    for c in (g.fwd, g.bwd):
        assert c.n_hub > 0 and c.band_plan is not None
    assert g.bwd.hub_w is not None
    S = g.num_slots
    x = X.int_tensor((n, 256), torch.bfloat16, seed=3, device=cuda_dev)
    gh = X.int_tensor((n * S, 256), torch.bfloat16, seed=4, device=cuda_dev)
    h_want = X.expected_csr_spmm(x, want.fwd, _lib.AGG_MEAN).view(n, S * 256)
    gx_want = X.expected_csr_spmm(gh, want.bwd, _lib.AGG_WEIGHTED)
    for graph in (g, g2):
        xg = x.clone().requires_grad_(True)
        h = G.rgcn_aggregate(xg, graph)
        assert torch.equal(h.detach().cpu(), h_want)
        h.backward(gh.view_as(h))
        assert torch.equal(xg.grad.cpu(), gx_want)
