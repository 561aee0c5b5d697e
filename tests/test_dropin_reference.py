"""Drop-in check against the REAL reference file, chungimungi/GMLM's ``main.py``, which is not part of
this repository: tests that use it run only where ``GMLM_REFERENCE_MAIN`` names a copy, and skip
otherwise.  They import that file unmodified with ``torch_geometric`` resolved to a shim that exposes
``gmlm_b200``'s ``RGCNConv`` / ``GraphNorm`` / ``degree`` (the import swap of INTEGRATION.md §1),
build the reference's own ``GraphTextLM`` with a stub PLM, and verify the state-dict ABI, the
optimiser grouping by parameter name and the reference's helpers that feed the path.  The NT-Xent
loss is also checked everywhere against vectors stored from the reference's own function
(tests/golden/nt_xent.npz)."""
import importlib.util
import os
import sys
import types
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.nn as nn

REF = Path(os.environ["GMLM_REFERENCE_MAIN"]) if os.environ.get("GMLM_REFERENCE_MAIN") else None
GOLDEN = Path(__file__).resolve().parent / "golden"


def _require_reference():
    if REF is None or not REF.exists():
        pytest.skip("GMLM_REFERENCE_MAIN does not name the reference's main.py")


class _StubPLM(nn.Module):
    base_model_prefix = "stub"

    def __init__(self, hidden=32):
        super().__init__()
        self.config = types.SimpleNamespace(hidden_size=hidden)
        self.emb = nn.Embedding(100, hidden)

    def gradient_checkpointing_enable(self):
        pass


def _import_reference(tmp_dir, conv_cls, norm_cls, degree_fn):
    class Data:  # minimal stand-in for torch_geometric.data.Data (main.py:20,814)
        def __init__(self, **kw):
            self.__dict__.update(kw)

        @property
        def num_nodes(self):
            return self.x.size(0)

    tg = types.ModuleType("torch_geometric")
    tg_nn = types.ModuleType("torch_geometric.nn")
    tg_nn.RGCNConv, tg_nn.GraphNorm = conv_cls, norm_cls               # the import swap (main.py:6)
    tg_utils = types.ModuleType("torch_geometric.utils")
    tg_utils.degree = degree_fn                                         # main.py:7
    tg_t = types.ModuleType("torch_geometric.transforms")
    tg_data = types.ModuleType("torch_geometric.data")
    tg_data.Data = Data
    tg.nn, tg.utils, tg.transforms, tg.data = tg_nn, tg_utils, tg_t, tg_data
    saved = {k: sys.modules.get(k) for k in ("torch_geometric", "torch_geometric.nn", "torch_geometric.utils",
                                             "torch_geometric.transforms", "torch_geometric.data")}
    sys.modules.update({"torch_geometric": tg, "torch_geometric.nn": tg_nn, "torch_geometric.utils": tg_utils,
                        "torch_geometric.transforms": tg_t, "torch_geometric.data": tg_data})
    cwd = os.getcwd()
    os.chdir(tmp_dir)                                    # main.py opens a log file in the cwd at import
    try:
        spec = importlib.util.spec_from_file_location("gmlm_reference_main", str(REF))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        os.chdir(cwd)
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    mod.AutoModel = types.SimpleNamespace(from_pretrained=lambda *a, **k: _StubPLM())
    mod.AutoTokenizer = types.SimpleNamespace(from_pretrained=lambda *a, **k: object())
    return mod


@pytest.fixture(scope="module")
def ref_main(tmp_path_factory):
    _require_reference()
    import gmlm_b200 as G
    return _import_reference(tmp_path_factory.mktemp("refrun"), G.RGCNConv, G.GraphNorm, G.degree)


@pytest.fixture(scope="module")
def ref_main_on_oracle(tmp_path_factory):
    """The same unmodified reference file with the ORACLE operators behind the PyG names: lets the
    reference's own encoder body (main.py:250-320) run on CPU."""
    _require_reference()
    from oracle import GraphNormRef, RGCNConvRef, degree_ref
    return _import_reference(tmp_path_factory.mktemp("refrun_oracle"), RGCNConvRef, GraphNormRef,
                             lambda index, num_nodes=None: degree_ref(index, num_nodes))


def test_reference_model_builds_on_our_modules(ref_main):
    import gmlm_b200 as G
    model = ref_main.GraphTextLM(gnn_in_channels=24, hidden_channels=8, num_classes=3, num_relations=5, num_bases=30,
                                 dropout_rate=0.5, model_name="stub", plm_max_length=16)
    assert isinstance(model.rgcn1, G.RGCNConv) and isinstance(model.gnorm1, G.GraphNorm)
    sd = model.state_dict()
    dims = [24, 8, 16, 32, 64]
    for k in range(4):
        assert sd[f"rgcn{k+1}.weight"].shape == (30, dims[k], dims[k + 1])      # basis weights (PyG ABI)
        assert sd[f"rgcn{k+1}.comp"].shape == (5, 30)
        assert sd[f"rgcn{k+1}.root"].shape == (dims[k], dims[k + 1])
        assert sd[f"rgcn{k+1}.bias"].shape == (dims[k + 1],)
        for p in ("weight", "bias", "mean_scale"):
            assert sd[f"gnorm{k+1}.{p}"].shape == (dims[k + 1],)
    # deepcopy/restore of the state dict, as main.py:623,644 does
    import copy
    model.load_state_dict(copy.deepcopy(model.state_dict()))
    # the reference's optimiser grouping by name substring (main.py:375-398)
    opt = ref_main.setup_optimizer(model, 1e-3, 1e-5, 1e-4, 0.01)
    n_graph = len(opt.param_groups[0]["params"])
    assert n_graph == 3 * 4 + 3 * 3 + 3 * 2          # rgcn1-3 (4 each) + gnorm1-3 (3 each) + residual_proj1-3 (2 each)


def test_reference_helpers_match_oracle_and_no_cpu_path(ref_main):
    from oracle import soft_masking_ref
    import gmlm_b200 as G
    x = torch.randn(12, 5)
    m = torch.rand(12) < 0.4
    t = torch.randn(1, 5)
    # the oracle's restatement of main.py:92-99 equals the reference function itself, bit for bit
    assert torch.equal(ref_main.soft_masking_gnn_input(x, m, t, beta=0.7), soft_masking_ref(x, m, t, 0.7))
    model = ref_main.GraphTextLM(gnn_in_channels=5, hidden_channels=4, num_classes=2, model_name="stub")
    ei = torch.randint(0, 12, (2, 30))
    with pytest.raises(Exception) as exc:      # CPU tensors: the swapped-in degree()/RGCNConv refuse, no fallback
        model.get_graph_embeddings(x, ei)
    assert "CUDA" in str(exc.value) or "cuda" in str(exc.value)
    assert isinstance(exc.value, (G.GmlmError, NotImplementedError, RuntimeError))


@pytest.mark.parametrize("n,e", [(40, 160), (1, 3), (25, 0)])
def test_oracle_encoder_is_pinned_by_the_reference_body(ref_main_on_oracle, n, e):
    """Pins oracle.EncoderRef (structure: which outputs feed the fusion, residual placement, N>1 gate,
    checkpointing) and the vectorised edge typing against the reference's own get_graph_embeddings
    (main.py:250-320) and its per-edge loop (main.py:253-267), executed from the real file."""
    from oracle import EncoderRef, edge_type_bucket_ref
    m = ref_main_on_oracle
    torch.manual_seed(0)
    fin, hid = 12, 4
    model = m.GraphTextLM(gnn_in_channels=fin, hidden_channels=hid, num_classes=3, num_relations=5, num_bases=30,
                          dropout_rate=0.5, model_name="stub").eval()
    enc = EncoderRef(fin, hid, 32, dropout_rate=0.5, use_checkpoint=True).eval()
    missing, unexpected = enc.load_state_dict(model.state_dict(), strict=False)
    assert missing == []                                        # every encoder parameter exists under the same name
    ei = torch.randint(0, n, (2, e))
    x = torch.randn(n, fin)
    captured = {}
    orig = model.rgcn1.forward

    def spy(xx, edge_index, edge_type):
        captured["edge_type"] = edge_type.clone()
        return orig(xx, edge_index, edge_type)

    model.rgcn1.forward = spy
    with torch.no_grad():
        want = model.get_graph_embeddings(x, ei)                # the reference's code, Python edge loop included
        got = enc(x, ei)
    assert torch.equal(captured["edge_type"], edge_type_bucket_ref(ei, n))
    assert torch.allclose(got, want, rtol=0, atol=1e-6)


# ----------------------------------------------------------------------------- §8f N4: NT-Xent consumer
@pytest.mark.parametrize("n,bs", [(0, 8), (1, 8), (8, 8), (9, 8), (10, 8), (37, 8), (64, 8), (23, 5), (12, None), (7, 16)])
def test_batched_nt_xent_equals_the_reference_function(ref_main_on_oracle, n, bs):
    """gmlm_b200.nt_xent_loss (one bmm over all chunks) against the reference's own chunk loop
    (main.py:102-136) on the same inputs: value and both input gradients, fp64."""
    from gmlm_b200.losses import nt_xent_loss
    g = torch.Generator().manual_seed(100 + n)
    z1 = torch.randn(n, 24, dtype=torch.float64, generator=g)
    z2 = torch.randn(n, 24, dtype=torch.float64, generator=g)
    a1, a2 = z1.clone().requires_grad_(True), z2.clone().requires_grad_(True)
    b1, b2 = z1.clone().requires_grad_(True), z2.clone().requires_grad_(True)
    want = ref_main_on_oracle.nt_xent_loss(a1, a2, temperature=0.5, batch_size=bs)
    got = nt_xent_loss(b1, b2, temperature=0.5, batch_size=bs)
    assert got.shape == want.shape and got.requires_grad == want.requires_grad
    assert abs(float(got) - float(want)) <= 1e-12 * max(1.0, abs(float(want)))
    if want.grad_fn is not None:
        want.backward()
        got.backward()
        assert torch.allclose(b1.grad, a1.grad, rtol=1e-11, atol=1e-13)
        assert torch.allclose(b2.grad, a2.grad, rtol=1e-11, atol=1e-13)
    else:
        assert float(got) == 0.0 and got.grad_fn is None


@pytest.mark.parametrize("case", range(5))
def test_batched_nt_xent_equals_the_stored_reference_vectors(case):
    """The same comparison without the reference file: gmlm_b200.nt_xent_loss in fp64 on CPU against the value
    and input gradients the reference's own nt_xent_loss gave on the stored inputs (tests/golden/nt_xent.npz,
    written by tests/golden/make_nt_xent_golden.py)."""
    from gmlm_b200.losses import nt_xent_loss
    z = np.load(GOLDEN / "nt_xent.npz")
    n, d, bs = z["cases"][case].tolist()
    b1 = torch.from_numpy(z[f"z1_{case}"]).double().requires_grad_(True)
    b2 = torch.from_numpy(z[f"z2_{case}"]).double().requires_grad_(True)
    assert b1.shape == b2.shape == (n, d)
    got = nt_xent_loss(b1, b2, temperature=float(z["temperature"][case]), batch_size=None if bs < 0 else bs)
    want = float(z[f"loss_{case}"])
    assert abs(float(got.detach()) - want) <= 1e-12 * max(1.0, abs(want))
    got.backward()
    assert torch.allclose(b1.grad, torch.from_numpy(z[f"g1_{case}"]), rtol=1e-11, atol=1e-13)
    assert torch.allclose(b2.grad, torch.from_numpy(z[f"g2_{case}"]), rtol=1e-11, atol=1e-13)


# ----------------------------------------------------------------------------- §8f N2: active-node mask sampler
@pytest.mark.parametrize("case", ["train_mask", "no_mask", "split_edge", "zero_degree", "empty_mask", "one_select"])
@pytest.mark.parametrize("seed", [0, 7])
def test_mask_sampler_is_bit_identical_to_the_reference(ref_main_on_oracle, case, seed):
    """gmlm_b200.generate_active_node_mask against the reference's own function (main.py:47-89) under the
    same seed: same branches, same random stream (multinomial == exponential race + topk) => same mask."""
    from types import SimpleNamespace
    from gmlm_b200.sampling import generate_active_node_mask
    from oracle import degree_ref
    ref = ref_main_on_oracle
    g = torch.Generator().manual_seed(seed)
    n, e = 400, 3000
    ei = torch.randint(0, n, (2, e), generator=g)
    x = torch.randn(n, 4, generator=g)
    kw, ratio = {}, 0.3
    train_mask = torch.rand(n, generator=g) < 0.6
    if case == "zero_degree":
        ei = ei[:, :0]
    if case == "empty_mask":
        train_mask = torch.zeros(n, dtype=torch.bool)
    if case == "one_select":
        ratio = 0.0                                             # num_select = max(1, 0) = 1 -> argmax branch
    data = SimpleNamespace(x=x, edge_index=ei, num_nodes=n, train_mask=train_mask)
    if case == "no_mask":
        data.train_mask = None
    if case == "split_edge":
        kw = {"split_edge": {"train": {"edge": ei[:, :500].t()}}, "base_mask_name": None}
    torch.manual_seed(100 + seed)
    want = ref.generate_active_node_mask(data, ratio, **kw)
    torch.manual_seed(100 + seed)
    got = generate_active_node_mask(data, ratio, deg=degree_ref(ei[0], n), **kw)
    assert got.dtype == torch.bool and torch.equal(got, want)
    if case not in ("empty_mask",):
        assert int(got.sum()) >= 1


def test_weighted_sampler_distribution_and_zero_weights():
    from gmlm_b200.sampling import weighted_sample_without_replacement
    w = torch.tensor([0.0, 1.0, 2.0, 0.0, 5.0, 0.5])
    g = torch.Generator().manual_seed(0)
    first = torch.zeros(6)
    for _ in range(4000):
        idx = weighted_sample_without_replacement(w, 3, g)
        assert idx.unique().numel() == 3 and not bool(((idx == 0) | (idx == 3)).any())     # zero weights never drawn
        first[idx[0]] += 1                                     # topk is sorted: idx[0] is the first draw
    p = w / w.sum()
    assert float((first / first.sum() - p).abs().max()) < 0.03   # first draw ~ weights


def test_batched_nt_xent_property(ref_main_on_oracle):
    """Random shapes / chunk sizes / temperatures: batched == reference loop (value and gradients)."""
    from hypothesis import given, settings, strategies as st
    from gmlm_b200.losses import nt_xent_loss
    ref = ref_main_on_oracle

    @settings(max_examples=40, deadline=None)
    @given(n=st.integers(0, 70), d=st.integers(1, 17), bs=st.one_of(st.none(), st.integers(1, 12)),
           temp=st.floats(0.05, 2.0), seed=st.integers(0, 10_000))
    def check(n, d, bs, temp, seed):
        g = torch.Generator().manual_seed(seed)
        z1 = torch.randn(n, d, dtype=torch.float64, generator=g) + 0.1
        z2 = torch.randn(n, d, dtype=torch.float64, generator=g) + 0.1
        a1, a2 = z1.clone().requires_grad_(True), z2.clone().requires_grad_(True)
        b1, b2 = z1.clone().requires_grad_(True), z2.clone().requires_grad_(True)
        want = ref.nt_xent_loss(a1, a2, temperature=temp, batch_size=bs)
        got = nt_xent_loss(b1, b2, temperature=temp, batch_size=bs)
        assert abs(float(got.detach()) - float(want.detach())) <= 1e-10 * max(1.0, abs(float(want.detach())))
        if want.grad_fn is not None:
            want.backward()
            got.backward()
            assert torch.allclose(b1.grad, a1.grad, rtol=1e-9, atol=1e-11)
            assert torch.allclose(b2.grad, a2.grad, rtol=1e-9, atol=1e-11)
        else:
            assert got.grad_fn is None

    check()


# ----------------------------------------------------------------------------- N3: ingest (main.py:780-837)
def _write_npz(path, n=57, e=300, f=9, classes=4, seed=0):
    import numpy as np
    rng = np.random.RandomState(seed)
    np.savez(path, node_features=rng.randn(n, f).astype(np.float32), edges=rng.randint(0, n, size=(2, e)),
             node_labels=rng.randint(0, classes, size=n), node_texts=np.array([f"text {i}" for i in range(n)], dtype=object),
             label_texts=np.array([f"label {c}" for c in range(classes)], dtype=object),
             train_masks=rng.rand(n) < 0.5, val_masks=rng.rand(n) < 0.3, test_masks=rng.rand(n) < 0.2)


def test_load_npz_graph_equals_the_reference_loader(ref_main, tmp_path):
    """gmlm_b200.load_npz_graph vs the reference's own load_npz_dataset on the same file, both split modes."""
    from gmlm_b200.ingest import load_npz_graph
    p = str(tmp_path / "toy.npz")
    _write_npz(p)
    for ratios in (None, (0.48, 0.32, 0.20), (0.5, 0.25, 0.25)):
        want, wf, wc = ref_main.load_npz_dataset("toy", p, split_ratios=ratios)
        got, gf, gc = load_npz_graph(p, split_ratios=ratios)
        assert (gf, gc) == (wf, wc)
        for k in ("x", "edge_index", "y", "train_mask", "val_mask", "test_mask"):
            a, b = getattr(got, k), getattr(want, k)
            assert a.dtype == b.dtype and torch.equal(a, b), k
        assert got.node_texts == want.node_texts and got.label_texts == want.label_texts


def test_augment_graph_keeps_the_same_edges_as_the_reference_under_a_seed(ref_main, tmp_path):
    from gmlm_b200.ingest import augment_graph, edge_dropout_mask, load_npz_graph
    p = str(tmp_path / "toy.npz")
    _write_npz(p, e=5000)
    want, _, _ = ref_main.load_npz_dataset("toy", p)
    got, _, _ = load_npz_graph(p)
    torch.manual_seed(7)
    want = ref_main.augment_graph(want, edge_dropout_p=0.1)
    torch.manual_seed(7)
    keep = edge_dropout_mask(got.edge_index.size(1), 0.1)
    torch.manual_seed(7)
    got = augment_graph(got, edge_dropout_p=0.1)
    assert torch.equal(got.edge_index, want.edge_index)
    assert int(keep.sum()) == want.edge_index.size(1) and 0.85 < keep.float().mean() < 0.95
