"""Transform-first RGCNConv (``gmlm_dst_plan`` + ``rgcn_transform_first``): the same layer as
[PyG] RGCNConv.forward (main.py:272) with the dense transform ahead of the gather, so that the [N, S*Fi]
matrix H is never materialised.  Checked against the fp64 oracle, against the aggregate-first formulation,
and — integers — against a numpy restatement of the plan."""
import numpy as np
import pytest
import torch

import gmlm_b200 as G
from gmlm_b200 import synth
from oracle import RGCNConvRef, edge_type_bucket_ref

from conftest import elementwise_err, rel_err

pytestmark = pytest.mark.gpu


def test_dst_plan_matches_numpy_restatement(cuda_dev):
    n, e = 700, 9000
    ei = synth.rmat_edges(n, e, seed=5)
    et = edge_type_bucket_ref(ei, n)
    g = G.RelGraph.build(ei.to(cuda_dev), et.to(cuda_dev), n, 5)
    S = g.num_slots
    f, b = g.dst_plan()
    rowptr = g.fwd.rowptr.cpu().numpy().astype(np.int64)
    col = g.fwd.col.cpu().numpy().astype(np.int64)
    want_rowptr = rowptr[::S][: n + 1] + np.arange(n + 1)
    assert np.array_equal(f.rowptr.cpu().numpy(), want_rowptr)
    want_col, want_w = [], []
    for i in range(n):
        for s in range(S):
            lo, hi = rowptr[i * S + s], rowptr[i * S + s + 1]
            want_col += list(col[lo:hi] * (S + 1) + s)
            if hi > lo:
                want_w += [np.float32(1.0) / np.float32(hi - lo)] * int(hi - lo)
        want_col.append(i * (S + 1) + S)
        want_w.append(np.float32(1.0))
    assert np.array_equal(f.col.cpu().numpy(), np.array(want_col, dtype=np.int32))
    assert np.array_equal(f.w.cpu().numpy(), np.array(want_w, dtype=np.float32))          # bit-exact weights
    # transposed plan: row r of dZ lists the destinations that gathered Z row r, with the same weights
    dense = torch.zeros(n, n * (S + 1), dtype=torch.float64)
    fr = f.rowptr.cpu().tolist()
    for i in range(n):
        for p in range(fr[i], fr[i + 1]):
            dense[i, want_col[p]] += float(want_w[p])
    dense_t = torch.zeros_like(dense.t())
    br, bc, bw = b.rowptr.cpu().tolist(), b.col.cpu().tolist(), b.w.cpu().tolist()
    assert b.num_rows == n * (S + 1)
    for r in range(b.num_rows):
        for p in range(br[r], br[r + 1]):
            dense_t[r, bc[p]] += bw[p]
    assert torch.equal(dense_t, dense.t().contiguous())


@pytest.mark.parametrize("n,e,fi,fo", [(183, 300, 1703, 64), (3000, 40000, 256, 64), (500, 6000, 96, 32),
                                      (500, 6000, 96, 22), (1, 2, 16, 8), (3000, 40000, 512, 128)])
def test_transform_first_fp32_matches_oracle_and_aggregate_first(cuda_dev, n, e, fi, fo):
    torch.manual_seed(1)
    ei = synth.rmat_edges(n, e, seed=n) if n > 1 else torch.zeros(2, e, dtype=torch.int64)
    et = edge_type_bucket_ref(ei, n)
    ref = RGCNConvRef(fi, fo, 5, 30).double()
    with torch.no_grad():
        ref.bias.uniform_(-0.1, 0.1)
    x, gout = torch.randn(n, fi), torch.randn(n, fo)
    x64 = x.double().requires_grad_(True)
    y_ref = ref(x64, ei, et)
    y_ref.backward(gout.double())
    outs = {}
    for tf in (True, False):
        mod = G.RGCNConv(fi, fo, 5, 30)
        mod.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
        mod = mod.to(cuda_dev)
        mod.transform_first = tf
        xg = x.to(cuda_dev).requires_grad_(True)
        y = mod(xg, ei.to(cuda_dev), et.to(cuda_dev))
        y.backward(gout.to(cuda_dev))
        assert y.dtype == torch.float32
        assert rel_err(y, y_ref) <= 1e-5 and elementwise_err(y, y_ref) <= 5e-4, tf
        assert rel_err(xg.grad, x64.grad) <= 1e-5, tf
        for name in ("weight", "comp", "root", "bias"):
            assert rel_err(getattr(mod, name).grad, getattr(ref, name).grad) <= 2e-5, (tf, name)
        assert torch.count_nonzero(mod.comp.grad[4]) == 0
        outs[tf] = y
    assert rel_err(outs[True], outs[False]) <= 1e-5


def test_transform_first_bf16_tcgen05_matches_oracle(cuda_dev):
    """The bandwidth-study input layer (256 -> 64, bf16): Z on the tcgen05 GEMM, 128-byte slab gather."""
    _bf16_transform_first_matches_oracle(cuda_dev, 256, 64)


def test_transform_first_bf16_tcgen05_512B_slabs_match_oracle(cuda_dev):
    """1024 -> 256, bf16: the gathered slabs are 512-byte rows, whose hub rows take the band plan (weighted, with
    hub_w)."""
    _bf16_transform_first_matches_oracle(cuda_dev, 1024, 256)


def _bf16_transform_first_matches_oracle(cuda_dev, fi, fo):
    n, e = 5000, 90000
    torch.manual_seed(0)
    ei = synth.rmat_edges(n, e, seed=3)
    et = edge_type_bucket_ref(ei, n)
    ref = RGCNConvRef(fi, fo, 5, 30).double()
    with torch.no_grad():
        ref.bias.uniform_(-0.1, 0.1)
    x, gout = torch.randn(n, fi).bfloat16(), torch.randn(n, fo).bfloat16()
    x64 = x.double().requires_grad_(True)
    y_ref = ref(x64, ei, et)
    y_ref.backward(gout.double())
    mod = G.RGCNConv(fi, fo, 5, 30, out_dtype=torch.bfloat16)
    mod.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    mod = mod.to(cuda_dev)
    assert mod._use_transform_first(G.get_rel_graph(ei.to(cuda_dev), et.to(cuda_dev), n, 5))   # chosen by the byte model
    xg = x.to(cuda_dev).requires_grad_(True)
    y = mod(xg, ei.to(cuda_dev), et.to(cuda_dev))
    y.backward(gout.to(cuda_dev))
    assert y.dtype == torch.bfloat16
    assert rel_err(y, y_ref) <= 2e-2 and rel_err(xg.grad, x64.grad) <= 2e-2
    for name in ("weight", "comp", "root", "bias"):
        assert rel_err(getattr(mod, name).grad, getattr(ref, name).grad) <= 2e-2, name
    # deterministic: same bits run to run (no atomics anywhere on the path)
    xg2 = x.to(cuda_dev).requires_grad_(True)
    y2 = mod(xg2, ei.to(cuda_dev), et.to(cuda_dev))
    y2.backward(gout.to(cuda_dev))
    assert torch.equal(y, y2) and torch.equal(xg.grad, xg2.grad)


def test_transform_first_on_a_partition_shaped_graph(cuda_dev):
    """num_src > num_nodes (destination-row partition: x = [local ‖ halo]); root term over the local rows."""
    n_dst, n_src, e, fi, fo = 400, 1000, 6000, 128, 32
    g = torch.Generator().manual_seed(7)
    src = torch.randint(0, n_src, (e,), generator=g)
    dst = torch.randint(0, n_dst, (e,), generator=g)
    et = torch.randint(0, 4, (e,), generator=g)
    ei = torch.stack([src, dst])
    graph = G.RelGraph.build(ei.to(cuda_dev), et.to(cuda_dev), n_dst, 5, num_src=n_src)
    mod = G.RGCNConv(fi, fo, 5, 30).to(cuda_dev)
    with torch.no_grad():
        mod.bias.uniform_(-0.1, 0.1)
    x = torch.randn(n_src, fi, generator=g).to(cuda_dev)
    gout = torch.randn(n_dst, fo, generator=g).to(cuda_dev)
    res = {}
    for tf in (True, False):
        mod.transform_first = tf
        mod.zero_grad()
        xg = x.clone().requires_grad_(True)
        y = mod(xg, graph)
        y.backward(gout)
        res[tf] = (y.detach(), xg.grad, mod.weight.grad.clone(), mod.root.grad.clone(), mod.bias.grad.clone())
    for a, b in zip(res[True], res[False]):
        assert rel_err(a, b) <= 1e-5


@pytest.mark.parametrize("mode", ["autocast", "bf16"])
@pytest.mark.parametrize("n,e,fi,fo", [(3000, 4500, 300, 512), (2000, 9000, 64, 128), (500, 200, 128, 256),
                                      (2000, 9000, 64, 22), (64, 0, 64, 64)])
def test_segment_compact_matches_dense_and_oracle(cuda_dev, mode, n, e, fi, fo):
    """The segment-compact formulation (one GEMM per populated relation over the non-empty (dst, rel) segments only,
    RelGraph.seg_plan) against the dense aggregate-first layer and the fp64 oracle: output, input gradient and every
    parameter gradient; sparse graphs like the reference's own (most segments empty), and a graph without edges."""
    torch.manual_seed(2)
    ei = synth.rmat_edges(n, e, seed=n + e) if e else torch.zeros(2, 0, dtype=torch.int64)
    et = edge_type_bucket_ref(ei, n)
    ref = RGCNConvRef(fi, fo, 5, 30).double()
    with torch.no_grad():
        ref.bias.uniform_(-0.1, 0.1)
    dt = torch.bfloat16 if mode == "bf16" else torch.float32
    x, gout = torch.randn(n, fi).to(dt), torch.randn(n, fo).to(dt)
    x64 = x.double().requires_grad_(True)
    y_ref = ref(x64, ei, et)
    y_ref.backward(gout.double())
    tol, gtol = (2e-2, 2e-2) if mode == "bf16" else (2e-3, 5e-3)
    outs = {}
    for compact in (True, False):
        mod = G.RGCNConv(fi, fo, 5, 30, out_dtype=dt if mode == "bf16" else None)
        mod.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
        mod = mod.to(cuda_dev)
        mod.segment_compact, mod.transform_first = compact, False
        xg = x.to(cuda_dev).requires_grad_(True)
        with torch.amp.autocast("cuda", enabled=mode == "autocast"):
            y = mod(xg, ei.to(cuda_dev), et.to(cuda_dev))
        y.backward(gout.to(cuda_dev).to(y.dtype))
        assert rel_err(y, y_ref) <= tol, compact
        assert rel_err(xg.grad, x64.grad, floor=1e-6) <= tol, compact
        for name in ("weight", "comp", "root", "bias"):
            assert rel_err(getattr(mod, name).grad, getattr(ref, name).grad, floor=1e-6) <= gtol, (compact, name)
        outs[compact] = y.float()
    assert rel_err(outs[True], outs[False]) <= tol


def test_seg_plan_structure(cuda_dev):
    """seg_plan: rows = the non-empty segments in slot-major order (slots start on multiples of 8 rows), edges in CSR
    order, destination of every row, transposed plan with 1/|segment| weights."""
    n, e = 700, 2000
    ei = synth.rmat_edges(n, e, seed=3)
    et = edge_type_bucket_ref(ei, n)
    g = G.RelGraph.build(ei.to(cuda_dev), et.to(cuda_dev), n, 5)
    p = g.seg_plan()
    S = g.num_slots
    rp = g.fwd.rowptr.cpu().long()
    lens = rp[1:] - rp[:-1]
    assert p.num_segments == int((lens > 0).sum()) == g.num_nonempty_segments
    rpc, colc, dstc = p.fwd.rowptr.cpu().long(), p.fwd.col.cpu(), p.dst.cpu()
    col = g.fwd.col.cpu()
    for s in range(S):
        a, c = p.slot_start[s], p.slot_count[s]
        assert a % 8 == 0
        segs = [d * S + s for d in range(n) if lens[d * S + s] > 0]
        assert c == len(segs)
        for k, seg in enumerate(segs[:50]):
            assert dstc[a + k] == seg // S
            assert torch.equal(colc[rpc[a + k]:rpc[a + k + 1]], col[rp[seg]:rp[seg + 1]])
    assert int(rpc[-1]) == e
    w = p.bwd.w.cpu()
    crow = p.bwd.col.cpu().long()
    assert torch.allclose(w, 1.0 / (rpc[crow + 1] - rpc[crow]).float())
