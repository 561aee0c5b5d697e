"""The band plan keyed on the use rank of the gathered rows (``CSR.col_rank`` / ``gmlm_col_rank``, the key
``plan_hubs`` builds the band plan on): the rank against a numpy restatement, the plan against the id-keyed
reference of test_gpu_spmm_hub_bands run on the ranks, and the aggregation that runs it against fp64, on R-MAT,
uniform and hand-built graphs."""
import numpy as np
import pytest
import torch

import gmlm_b200 as G
from gmlm_b200 import _lib, synth
from gmlm_b200.graph import HUB_BAND_MIN_RUN, HUB_BAND_SHIFT

from conftest import rel_err
from test_gpu_spmm_hub_bands import _ref, _without_bands, plan_ref

pytestmark = pytest.mark.gpu


def rank_ref(col, num_cols):
    count = np.bincount(col, minlength=num_cols)
    order = np.lexsort((np.arange(num_cols), -count))          # count desc, then id asc
    rank = np.empty(num_cols, np.int64)
    rank[order] = np.arange(num_cols)
    return rank


def _check(csr, shift):
    """The plan of `csr` with the rank key at `shift`, integer-exact against plan_ref on rank[col]."""
    rp = csr.rowptr.cpu().numpy().astype(np.int64)
    col = csr.col.cpu().numpy().astype(np.int64)
    rank = csr.col_rank().cpu().numpy().astype(np.int64)
    assert rank.size == col.max() + 1
    np.testing.assert_array_equal(rank, rank_ref(col, rank.size))
    csr.plan_bands(shift, rank=csr.col_rank())
    w = csr.w.cpu().numpy() if csr.w is not None else None
    # rank is a permutation, so ordering edges by rank[col] is ordering them by col's rank
    hub_key, hub_w, chunk_ptr, cut, order = plan_ref(rp, rank[col], w, csr.hub_thresh, shift, HUB_BAND_MIN_RUN)
    nh, nb = csr.n_hub, csr.n_band_chunks
    hub_col = csr.hub_col.cpu().numpy().astype(np.int64)
    bp = csr.band_plan.cpu().numpy().astype(np.int64)
    assert bp.size == nh + 2 + 2 * nb
    np.testing.assert_array_equal(rank[hub_col], hub_key)
    if w is not None:
        np.testing.assert_array_equal(csr.hub_w.cpu().numpy(), hub_w)
    np.testing.assert_array_equal(bp[:nh + 1], chunk_ptr)
    np.testing.assert_array_equal(bp[nh + 1:nh + 2 + nb], cut)
    np.testing.assert_array_equal(bp[nh + 2 + nb:], order)
    # each hub row's edges exactly once, rank non-decreasing inside a row, chunks inside one row and <= hub_thresh
    hub_rows = csr.hub_row.cpu().numpy()
    off = np.concatenate([[0], np.cumsum(rp[hub_rows + 1] - rp[hub_rows])])
    for h, r in enumerate(hub_rows):
        a, b = off[h], off[h + 1]
        np.testing.assert_array_equal(np.sort(hub_col[a:b]), np.sort(col[rp[r]:rp[r + 1]]))
        assert np.all(np.diff(rank[hub_col[a:b]]) >= 0)
        c = cut[chunk_ptr[h]:chunk_ptr[h + 1] + 1]
        assert c[0] == a and c[-1] == b and np.all(np.diff(c) >= 1) and np.all(np.diff(c) <= csr.hub_thresh)
    band = rank[hub_col[cut[:-1]]] >> shift
    assert np.all(np.diff(band[order]) >= 0)                  # chunks launched band by band
    return nb


def _hand_csr(rows, dev, thresh=64, w=None):
    rowptr = np.zeros(len(rows) + 1, np.int64)
    rowptr[1:] = np.cumsum([len(r) for r in rows])
    col = np.concatenate([np.asarray(r, np.int64) for r in rows if len(r)])
    csr = G.graph.CSR(rowptr=torch.tensor(rowptr, dtype=torch.int32, device=dev),
                      col=torch.tensor(col, dtype=torch.int32, device=dev), num_rows=len(rows), hub_thresh=thresh,
                      w=None if w is None else torch.tensor(w, dtype=torch.float32, device=dev))
    return csr.plan_hubs()


def _hand_rows(case):
    rng = np.random.default_rng(1)
    if case == "all_edges_one_row":
        return [[], list(rng.integers(0, 500, 300)), []]
    if case == "ties":                   # every gathered row used equally often: rank = id order
        return [list(rng.permutation(np.tile(np.arange(40), 5))) for _ in range(3)]
    if case == "empty_rows":
        return [[], [], list(rng.integers(0, 50, 200)), [], list(rng.integers(0, 50, 3)), []]
    if case == "single_hub_row":
        return [list(rng.integers(0, 1000, 8)) for _ in range(20)] + [list(rng.zipf(1.5, 700) % 1000)]
    if case == "all_hub":
        return [list(rng.zipf(1.3, int(rng.integers(65, 400))) % 3000) for _ in range(12)]
    raise ValueError(case)


@pytest.mark.parametrize("case", ["all_edges_one_row", "ties", "empty_rows", "single_hub_row", "all_hub"])
@pytest.mark.parametrize("shift", [2, 5])
def test_rank_plan_hand_built(cuda_dev, case, shift):
    csr = _hand_csr(_hand_rows(case), cuda_dev)
    assert csr.n_hub >= 1
    _check(csr, shift)
    if case == "ties":
        np.testing.assert_array_equal(csr.col_rank().cpu().numpy(), np.arange(40))


def test_rank_of_unused_rows_and_bad_index(cuda_dev):
    col = torch.tensor([5, 5, 2, 9, 2, 5], dtype=torch.int32, device=cuda_dev)
    csr = G.graph.CSR(rowptr=torch.tensor([0, 6], dtype=torch.int32, device=cuda_dev), col=col, num_rows=1)
    assert csr.col_rank().tolist() == [3, 4, 1, 5, 6, 0, 7, 8, 9, 2]   # 5 (x3), 2 (x2), 9, then unused ids
    lib = _lib.load()
    ws_bytes = lib.gmlm_col_rank_workspace_bytes(4)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=cuda_dev)
    rank = torch.empty(4, dtype=torch.int32, device=cuda_dev)
    rc = lib.gmlm_col_rank(col.data_ptr(), 6, 4, rank.data_ptr(), ws.data_ptr(), ws_bytes,
                           torch.cuda.current_stream().cuda_stream)
    assert rc != 0 and b"col_rank" in lib.gmlm_last_error()


@pytest.mark.parametrize("kind", ["rmat", "uniform"])
@pytest.mark.parametrize("shift", [6, 10, HUB_BAND_SHIFT])
def test_rank_plan_matches_numpy(cuda_dev, kind, shift):
    n, e = 20_000, 400_000
    ei = (synth.rmat_edges if kind == "rmat" else synth.uniform_edges)(n, e, seed=5).cuda()
    g = G.RelGraph.build(ei, G.edge_type_from_degree(ei, n), n, 5, hub_thresh=64 if kind == "rmat" else 16)
    for csr in (g.fwd, g.bwd):
        assert csr.n_hub > 0
        _check(csr, shift)


def test_default_plan_is_rank_keyed(cuda_dev):
    ei = synth.rmat_edges(20_000, 400_000, seed=5).cuda()
    g = G.RelGraph.build(ei, G.edge_type_from_degree(ei, 20_000), 20_000, 5, hub_thresh=64)
    for csr in (g.fwd, g.bwd):
        built = (csr.hub_col.clone(), csr.band_plan.clone())
        csr.plan_bands(HUB_BAND_SHIFT, rank=csr.col_rank())
        assert torch.equal(built[0], csr.hub_col) and torch.equal(built[1], csr.band_plan)


@pytest.fixture(scope="module")
def multi_band_graph(cuda_dev):
    """300k nodes, hub threshold 32: most edges on the hub path, gathered rows in several rank bands."""
    ei = synth.rmat_edges(300_000, 3_000_000, seed=11).cuda()
    return G.RelGraph.build(ei, G.edge_type_from_degree(ei, 300_000), 300_000, 5, hub_thresh=32)


@pytest.mark.parametrize("dtype,feat", [(torch.bfloat16, 256), (torch.float32, 128)])
def test_rank_banded_aggregation_fp64(multi_band_graph, dtype, feat):
    g = multi_band_graph
    n, S = g.num_nodes, g.num_slots
    x = synth.make_features(n, feat, device="cuda", seed=1, dtype=dtype)
    gh = synth.make_features(n * S, feat, device="cuda", seed=2, dtype=dtype)
    tol = 2e-2 if dtype == torch.bfloat16 else 1e-5
    for csr, inp, mode in ((g.fwd, x, _lib.AGG_MEAN), (g.bwd, gh, _lib.AGG_WEIGHTED)):
        assert (csr.col_rank().long()[csr.hub_col.long()] >> HUB_BAND_SHIFT).max() >= 1   # several rank bands
        out = G.spmm(inp, csr, mode)
        assert rel_err(out, _ref(inp.double(), csr, mode)) < tol
        assert torch.equal(out, G.spmm(inp, csr, mode))                 # run to run: bit-identical
        plain = G.spmm(inp, _without_bands(csr), mode)
        hub = torch.zeros(csr.num_rows, dtype=torch.bool, device=out.device)
        hub[csr.hub_row.long()] = True
        assert torch.equal(out[~hub], plain[~hub])                      # the rows kernel's rows, bit for bit
        assert rel_err(out[hub], plain[hub]) < tol
