"""GPU: GAT edge features, from the fused kernels' per-edge score term up to the GAT encoder over edge types.

* the kernels with ``a_edge`` against autograd of an fp64 softmax: fp32 and bf16 z, rows in one warp and rows cut
  into head groups (2048 and 4096 features), a hub row of more than 256 edges, duplicate edges and self-loops, with
  ``d_score`` checked as the gradient of ``a_edge``; the same under the hash dropout mask; bit-identical reruns;
* the loop fill (``gat_edge_scores``) against upstream's remove / add-self-loops with ``fill_value="mean"``;
* ``GATConv(edge_dim)`` against ``GATConvEdgeRef`` in fp64 (output and every gradient), fp32 and under autocast,
  with 1-D, one-hot and dense ``edge_attr``;
* ``GraphEncoder(conv="gat", gat_edge_types=True)`` against ``TypedGATEncoderRef``: fp32, autocast at
  hidden_channels = 512, the state-dict round trip, checkpointing with soft masking, ``GraphedEncoderStep`` replay,
  and exact-zero gradients for relation 4, which the degree buckets never produce."""
import copy

import pytest
import torch
import torch.nn.functional as F

import gmlm_b200 as G
from gmlm_b200 import synth
from gmlm_b200.attn import LoopGraph, gat_aggregate, gat_dropout_mask, gat_edge_scores
from oracle import soft_masking_ref

from conftest import rel_err
from gat_edge_ref import GATConvEdgeRef, TypedGATEncoderRef, loop_fill_mean_ref
from test_gat_edge_attr_cpu import KA_ATTR, KA_EDGES, KA_WANT, KA_X, ka_params

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
BF16_TOL = 2e-2


def _edges(n, e, seed):
    """uniform edges with self-loops and duplicates, plus a star of n + 40 edges into node 7: a hub row longer than
    the default hub threshold of 256.  With e ~ 2n, many nodes have no in-edge besides their own loop."""
    ei = synth.uniform_edges(n, e, seed=seed)
    ei[1, : e // 20] = ei[0, : e // 20]                             # self-loops (dropped, then one added per node)
    ei[:, e // 20: e // 10] = ei[:, e // 10: 3 * e // 20]           # duplicate edges
    star = torch.stack([torch.arange(n), torch.full((n,), 7)])
    return torch.cat([ei, star, star[:, :40]], dim=1)


def _reference(graph, z, a_s, a_d, a_e, keep=None, p=0.0, slope=0.2):
    """fp64 two-pass edge softmax in forward-CSR order with the edge term, differentiable in z, a_src, a_dst, a_edge"""
    rowptr, col = graph.fwd.rowptr.cpu().long(), graph.fwd.col.cpu().long()
    n, heads = a_d.shape
    c = z.size(1) // heads
    dst = torch.repeat_interleave(torch.arange(n), rowptr[1:] - rowptr[:-1])
    sc = F.leaky_relu(a_s[col] + a_d[dst] + a_e, slope)
    emax = torch.full((n, heads), float("-inf"), dtype=torch.float64).scatter_reduce(
        0, dst.unsqueeze(-1).expand_as(sc), sc.detach(), reduce="amax", include_self=True)
    ex = (sc - emax[dst]).exp()
    alpha = ex / (torch.zeros((n, heads), dtype=torch.float64).index_add_(0, dst, ex) + 1e-16)[dst]
    if keep is not None:
        alpha = alpha * keep.cpu().double() / (1.0 - p)
    out = torch.zeros((n, heads, c), dtype=torch.float64).index_add_(0, dst, alpha.unsqueeze(-1) * z.view(n, heads, c)[col])
    return out.view(n, heads * c)


@pytest.fixture(scope="module")
def hub_graph(cuda_dev):
    n = 700
    ei = _edges(n, 1500, seed=31).to(cuda_dev)
    graph = LoopGraph.build(ei, n)
    rows = graph.fwd.rowptr[1:] - graph.fwd.rowptr[:-1]
    assert int(rows.max()) > 256 and graph.fwd.n_hub >= 1 and graph.fwd.n_chunks > graph.fwd.n_hub
    assert int((rows == 1).sum()) > 0                               # nodes whose only entry is their loop
    return n, ei, graph


# (heads, head_dim): one warp; 2048 and 4096 features in head groups; odd widths on the scalar path, in groups
WIDTHS = [(8, 16), (8, 256), (8, 512), (3, 130)]


def _operands(graph, n, heads, c, dtype, seed):
    gen = torch.Generator().manual_seed(seed)
    z = torch.randn(n, heads * c, generator=gen).to(dtype)
    a_s = torch.randn(n, heads, generator=gen) * 2
    a_d = torch.randn(n, heads, generator=gen) * 2
    a_e = torch.randn(graph.fwd.nnz, heads, generator=gen) * 2
    gout = torch.randn(n, heads * c, generator=gen).to(dtype)
    return z, a_s, a_d, a_e, gout


def _run(dev, graph, z, a_s, a_d, a_e, gout, p=0.0, seed=0):
    leaves = [t.to(dev).requires_grad_(True) for t in (z, a_s, a_d, a_e)]
    out = gat_aggregate(leaves[0], leaves[1], leaves[2], graph, 0.2, p, seed, a_edge=leaves[3])
    out.backward(gout.to(dev))
    return out, [t.grad for t in leaves]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("heads,c", WIDTHS)
def test_kernels_with_edge_term_match_fp64_softmax(cuda_dev, hub_graph, heads, c, dtype):
    n, _, graph = hub_graph
    z, a_s, a_d, a_e, gout = _operands(graph, n, heads, c, dtype, heads * 1000 + c)
    out, grads = _run(cuda_dev, graph, z, a_s, a_d, a_e, gout)
    assert out.dtype == dtype
    ref_leaves = [t.double().requires_grad_(True) for t in (z, a_s, a_d, a_e)]
    ref = _reference(graph, *ref_leaves)
    ref.backward(gout.double())
    tol, gtol = (FP32_TOL, 2e-5) if dtype == torch.float32 else (BF16_TOL, BF16_TOL)
    assert rel_err(out, ref) <= tol
    for name, got, want in zip(("z", "a_src", "a_dst", "a_edge"), grads, ref_leaves):
        assert rel_err(got, want.grad) <= gtol, name
    # the term moves the result: the same call without it differs
    assert not torch.equal(out, gat_aggregate(z.to(cuda_dev), a_s.to(cuda_dev), a_d.to(cuda_dev), graph))
    # no atomics: a rerun is bit-identical, forward and backward
    out2, grads2 = _run(cuda_dev, graph, z, a_s, a_d, a_e, gout)
    assert torch.equal(out, out2)
    assert all(torch.equal(a, b) for a, b in zip(grads, grads2))


@pytest.mark.parametrize("heads,c", [(8, 16), (8, 512)])
def test_edge_term_applies_the_hash_dropout_mask(cuda_dev, hub_graph, heads, c):
    n, _, graph = hub_graph
    p, seed = 0.5, 987654321
    z, a_s, a_d, a_e, gout = _operands(graph, n, heads, c, torch.float32, c + 5)
    keep = gat_dropout_mask(seed, graph.fwd.nnz, heads, p, cuda_dev)
    out, grads = _run(cuda_dev, graph, z, a_s, a_d, a_e, gout, p, seed)
    ref_leaves = [t.double().requires_grad_(True) for t in (z, a_s, a_d, a_e)]
    ref = _reference(graph, *ref_leaves, keep=keep, p=p)
    ref.backward(gout.double())
    assert rel_err(out, ref) <= FP32_TOL
    for name, got, want in zip(("z", "a_src", "a_dst", "a_edge"), grads, ref_leaves):
        assert rel_err(got, want.grad) <= 2e-5, name
    out2, grads2 = _run(cuda_dev, graph, z, a_s, a_d, a_e, gout, p, seed)
    assert torch.equal(out, out2) and all(torch.equal(a, b) for a, b in zip(grads, grads2))


def test_loop_fill_matches_upstream_mean(cuda_dev, hub_graph):
    """gat_edge_scores: input self-loops dropped, each node's loop = the mean over its kept in-edges (0 without),
    in forward-CSR order; and the gradient of that map."""
    n, ei, graph = hub_graph
    heads = 3
    gen = torch.Generator().manual_seed(4)
    alpha = torch.randn(ei.size(1), heads, generator=gen)
    g = torch.randn(graph.fwd.nnz, heads, generator=gen)
    ag = alpha.to(cuda_dev).requires_grad_(True)
    a_edge = gat_edge_scores(ag, graph)
    a_edge.backward(g.to(cuda_dev))
    a64 = alpha.double().requires_grad_(True)
    _, filled = loop_fill_mean_ref(ei.cpu().long(), a64, n)       # kept edges, then loops 0..n-1: fwd.perm's order
    want = filled[graph.fwd.perm.cpu().long()]
    want.backward(g.double())
    assert rel_err(a_edge, want) <= 1e-6
    assert rel_err(ag.grad, a64.grad) <= 1e-6
    loops = ei[0] == ei[1]
    assert bool((ag.grad[loops] == 0).all())                      # a dropped input loop gets no gradient
    a2 = gat_edge_scores(ag.detach(), graph)
    assert torch.equal(a_edge.detach(), a2)


# ------------------------------------------------------------------------------------------------------- GATConv
def _edge_attr(kind, e, gen):
    if kind == "1d":
        return torch.randn(e, generator=gen)
    if kind == "onehot":
        return F.one_hot(torch.randint(0, 5, (e,), generator=gen), 5).float()
    return torch.randn(e, 16, generator=gen)


EDGE_DIM = {"1d": 1, "onehot": 5, "dense": 16}
PARAMS = ("lin.weight", "att_src", "att_dst", "lin_edge.weight", "att_edge", "bias")


def _conv_pair(fi, c, heads, d):
    ref = GATConvEdgeRef(fi, c, heads=heads, edge_dim=d).double()
    with torch.no_grad():
        ref.bias.uniform_(-0.1, 0.1)
    mod = G.GATConv(fi, c, heads=heads, edge_dim=d)
    assert set(mod.state_dict()) == set(ref.state_dict()) == set(PARAMS)
    mod.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    return ref, mod


def test_gat_conv_edge_attr_known_answer(cuda_dev):
    mod = G.GATConv(1, 1, heads=1, edge_dim=1).eval()
    mod.load_state_dict({k: v.float() for k, v in ka_params().items()})
    mod = mod.to(cuda_dev)
    out = mod(torch.tensor(KA_X, device=cuda_dev), torch.tensor(KA_EDGES, device=cuda_dev),
              torch.tensor(KA_ATTR, device=cuda_dev))
    assert torch.allclose(out.double().cpu(), torch.tensor(KA_WANT, dtype=torch.float64), rtol=FP32_TOL, atol=FP32_TOL)


@pytest.mark.parametrize("kind", ["1d", "onehot", "dense"])
@pytest.mark.parametrize("n,e,fi,c,heads", [(183, 300, 64, 16, 4), (2449, 9305, 300, 64, 8)])
def test_gat_conv_edge_attr_matches_oracle_fp32(cuda_dev, n, e, fi, c, heads, kind):
    torch.manual_seed(3)
    gen = torch.Generator().manual_seed(n + e)
    ei = _edges(n, e, seed=n + 7)
    ref, mod = _conv_pair(fi, c, heads, EDGE_DIM[kind])
    mod = mod.to(cuda_dev)
    x, ea, gout = torch.randn(n, fi, generator=gen), _edge_attr(kind, ei.size(1), gen), torch.randn(n, heads * c)
    x64, ea64 = x.double().requires_grad_(True), ea.double().requires_grad_(True)
    y_ref = ref(x64, ei, ea64)
    y_ref.backward(gout.double())
    xg, eag = x.to(cuda_dev).requires_grad_(True), ea.to(cuda_dev).requires_grad_(True)
    y = mod(xg, ei.to(cuda_dev), eag)
    y.backward(gout.to(cuda_dev))
    assert rel_err(y, y_ref) <= FP32_TOL
    assert rel_err(xg.grad, x64.grad) <= 2e-5
    assert rel_err(eag.grad, ea64.grad) <= 2e-5
    got, want = dict(mod.named_parameters()), dict(ref.named_parameters())
    for name in PARAMS:                      # the floor: see test_gpu_modules.test_gat_conv_matches_oracle
        assert rel_err(got[name].grad, want[name].grad, floor=1e-2) <= 2e-5, name
    # a LoopGraph passed in place of edge_index carries the same maps
    y2 = mod(xg.detach(), G.get_loop_graph(ei.to(cuda_dev), n), eag.detach())
    assert torch.equal(y.detach(), y2)
    # edge_attr=None is the layer without edge features
    plain = G.GATConv(fi, c, heads=heads).to(cuda_dev)
    plain.load_state_dict({k: v for k, v in mod.state_dict().items() if "edge" not in k})
    assert torch.equal(mod(xg.detach(), ei.to(cuda_dev)), plain(xg.detach(), ei.to(cuda_dev)))


@pytest.mark.parametrize("heads,c,kind", [(8, 64, "dense"), (8, 512, "onehot")])
def test_gat_conv_edge_attr_autocast_matches_oracle(cuda_dev, heads, c, kind):
    """Gates as in test_gpu_gat_encoder.test_gat_conv_autocast_matches_oracle: output at 2e-3, gradients at
    max(layer gate, 3x the error of the fp64 oracle fed the same fp16-rounded x and W).  The edge term is fp32."""
    torch.manual_seed(13)
    n, e, fi = 700, 6000, 300
    gen = torch.Generator().manual_seed(c)
    ei = _edges(n, e, seed=c)
    ref, mod = _conv_pair(fi, c, heads, EDGE_DIM[kind])
    mod = mod.to(cuda_dev)
    x, ea, gout = torch.randn(n, fi, generator=gen), _edge_attr(kind, ei.size(1), gen), torch.randn(n, heads * c)
    x64, ea64 = x.double().requires_grad_(True), ea.double().requires_grad_(True)
    y_ref = ref(x64, ei, ea64)
    y_ref.backward(gout.double())
    ref16 = copy.deepcopy(ref)                                    # the same oracle on fp16-rounded operands
    with torch.no_grad():
        ref16.lin.weight.copy_(ref.lin.weight.half().double())
    ref16.zero_grad()
    x16, ea16 = x.half().double().requires_grad_(True), ea.double().requires_grad_(True)
    ref16(x16, ei, ea16).backward(gout.double())
    xg, eag = x.to(cuda_dev).requires_grad_(True), ea.to(cuda_dev).requires_grad_(True)
    with torch.amp.autocast("cuda"):
        y = mod(xg, ei.to(cuda_dev), eag)
    assert y.dtype == torch.float32
    y.backward(gout.to(cuda_dev))
    assert rel_err(y, y_ref) <= 2e-3
    for got, want, want16 in ((xg.grad, x64.grad, x16.grad), (eag.grad, ea64.grad, ea16.grad)):
        noise = rel_err(want16, want)
        assert rel_err(got, want) <= max(2e-3, 3.0 * noise), noise
    for name in PARAMS:
        got = dict(mod.named_parameters())[name].grad
        want, want16 = dict(ref.named_parameters())[name].grad, dict(ref16.named_parameters())[name].grad
        noise = rel_err(want16, want, floor=1e-2)
        assert rel_err(got, want, floor=1e-2) <= max(5e-3, 3.0 * noise), (name, noise)


def test_gat_conv_edge_attr_dropout_is_reproducible(cuda_dev):
    n, e, fi, c, heads = 1500, 20000, 32, 16, 8
    ei = synth.rmat_edges(n, e, seed=9).to(cuda_dev)
    torch.manual_seed(1)
    mod = G.GATConv(fi, c, heads=heads, dropout=0.4, edge_dim=5).to(cuda_dev).train()
    x = torch.randn(n, fi, device=cuda_dev)
    ea = F.one_hot(torch.randint(0, 5, (ei.size(1),), device=cuda_dev), 5).float()
    y1, y2 = mod(x, ei, ea, dropout_seed=77), mod(x, ei, ea, dropout_seed=77)
    assert torch.equal(y1, y2) and not torch.equal(y1, mod(x, ei, ea, dropout_seed=78))
    assert not torch.equal(y1, mod(x, ei, dropout_seed=77))       # the edge term is applied under dropout too
    mod.eval()
    assert torch.equal(mod(x, ei, ea), mod(x, ei, ea))


# ------------------------------------------------------------------------------------------------ the typed encoder
def _typed_pair(fin, hidden, out_dim, heads, use_checkpoint=False):
    torch.manual_seed(5)
    ref = TypedGATEncoderRef(fin, hidden, out_dim, heads=heads, dropout_rate=0.0, use_checkpoint=False).double()
    with torch.no_grad():
        for k in range(1, 5):
            getattr(ref, f"gnorm{k}").mean_scale.uniform_(0.5, 1.0)
            getattr(ref, f"gat{k}").bias.uniform_(-0.1, 0.1)
    mod = G.GraphEncoder(fin, hidden, out_dim, dropout_rate=0.0, conv="gat", heads=heads, gat_edge_types=True,
                         use_checkpoint=use_checkpoint)
    keys = set(mod.state_dict())
    assert keys == set(ref.state_dict()) | {"gnn_mask_token_embed"}
    assert {f"gat{k}.{p}" for k in range(1, 5) for p in ("lin_edge.weight", "att_edge")} <= keys
    missing, unexpected = mod.load_state_dict({k: v.float() for k, v in ref.state_dict().items()}, strict=False)
    assert unexpected == [] and missing == ["gnn_mask_token_embed"]
    return ref, mod


def _relation4_grads_are_zero(mod):
    for k in range(1, 5):
        g = getattr(mod, f"gat{k}").lin_edge.weight.grad
        assert g is not None and int(torch.count_nonzero(g[:, 4])) == 0, k
        assert int(torch.count_nonzero(g[:, :4])) > 0, k


@pytest.mark.parametrize("n,e,fin,hidden,heads", [(183, 300, 64, 16, 4), (2000, 9000, 300, 16, 8)])
def test_typed_gat_encoder_matches_oracle_fp32(cuda_dev, n, e, fin, hidden, heads):
    ref, mod = _typed_pair(fin, hidden, 48, heads)
    mod = mod.to(cuda_dev)
    ei = _edges(n, e, seed=n + 3)
    x = torch.randn(n, fin)
    fused_ref = ref(x.double(), ei)
    fused = mod.get_graph_embeddings(x.to(cuda_dev), ei.to(cuda_dev))
    assert rel_err(fused, fused_ref) <= FP32_TOL
    gout = torch.randn(n, 48)
    fused_ref.backward(gout.double())
    fused.backward(gout.to(cuda_dev))
    ref32 = copy.deepcopy(ref).float()                            # the fp32 oracle's own error: the gradient yardstick
    ref32.zero_grad()
    ref32(x, ei).backward(gout)
    sd_ref, sd32 = dict(ref.named_parameters()), dict(ref32.named_parameters())
    for name, p in mod.named_parameters():
        if name == "gnn_mask_token_embed":
            continue
        if sd_ref[name].grad is None:                             # residual_proj3 is dead (main.py:317-318)
            assert p.grad is None, name
            continue
        noise = rel_err(sd32[name].grad, sd_ref[name].grad, floor=1e-2)
        assert rel_err(p.grad, sd_ref[name].grad, floor=1e-2) <= max(2e-5, 3.0 * noise), (name, noise)
    _relation4_grads_are_zero(mod)
    # the typed encoder differs from the untyped one with the same shared weights
    plain = G.GraphEncoder(fin, hidden, 48, dropout_rate=0.0, conv="gat", heads=heads).to(cuda_dev)
    plain.load_state_dict({k: v for k, v in mod.state_dict().items() if "edge" not in k})
    with torch.no_grad():
        assert not torch.equal(plain.get_graph_embeddings(x.to(cuda_dev), ei.to(cuda_dev)), fused.detach())


def test_typed_gat_encoder_autocast_at_amazon_ratings_scale(cuda_dev):
    n, e, fin, hidden = 2449, 9305, 300, 512
    ref, mod = _typed_pair(fin, hidden, 768, 8)
    mod = mod.to(cuda_dev)
    ref = ref.to(cuda_dev)                                        # fp64 reference on the GPU (4096-wide layers)
    ei = _edges(n, e, seed=17).to(cuda_dev)
    x = torch.randn(n, fin, device=cuda_dev)
    with torch.no_grad():
        fused_ref = ref(x.double(), ei)
    with torch.amp.autocast("cuda"):
        fused = mod.get_graph_embeddings(x, ei)
    assert fused.dtype == torch.float32
    assert rel_err(fused, fused_ref) <= BF16_TOL
    fused.backward(torch.randn_like(fused))
    for name, p in mod.named_parameters():
        if name in ("gnn_mask_token_embed", "residual_proj3.weight", "residual_proj3.bias"):
            assert p.grad is None, name
            continue
        assert p.grad is not None and bool(torch.isfinite(p.grad).all()), name
    _relation4_grads_are_zero(mod)


def test_typed_gat_encoder_state_dict_round_trip(cuda_dev):
    ref, mod = _typed_pair(64, 16, 32, 4)
    sd = {k: v for k, v in mod.state_dict().items() if k != "gnn_mask_token_embed"}
    back = TypedGATEncoderRef(64, 16, 32, heads=4, dropout_rate=0.0, use_checkpoint=False).double()
    back.load_state_dict({k: v.double() for k, v in sd.items()})          # strict: every key, every shape
    for k, v in ref.state_dict().items():
        assert torch.equal(back.state_dict()[k], v.float().double()), k
    mod2 = G.GraphEncoder(64, 16, 32, dropout_rate=0.0, conv="gat", heads=4, gat_edge_types=True).to(cuda_dev)
    mod2.load_state_dict(mod.state_dict())
    ei = _edges(300, 600, seed=2).to(cuda_dev)
    x = torch.randn(300, 64, device=cuda_dev)
    with torch.no_grad():
        assert torch.equal(mod.to(cuda_dev).get_graph_embeddings(x, ei), mod2.get_graph_embeddings(x, ei))


def test_typed_gat_encoder_soft_mask_with_checkpointing(cuda_dev):
    n, e, fin, hidden, heads = 600, 3000, 64, 16, 4
    ref, mod = _typed_pair(fin, hidden, 32, heads, use_checkpoint=True)
    mod = mod.to(cuda_dev)
    plain = copy.deepcopy(mod)
    plain.use_checkpoint = False
    ei = _edges(n, e, seed=77).to(cuda_dev)
    gen = torch.Generator().manual_seed(8)
    x = torch.randn(n, fin, generator=gen)
    mask = torch.rand(n, generator=gen) < 0.3
    tok = mod.gnn_mask_token_embed.detach().cpu()
    fused_ref = ref(soft_masking_ref(x.double(), mask, tok.double()), ei.cpu())
    gout = torch.randn(n, 32, generator=gen).to(cuda_dev)
    xs = [x.to(cuda_dev).requires_grad_(True) for _ in range(2)]
    outs = []
    for m, xg in zip((mod, plain), xs):
        y = m(xg, ei, gnn_perturb_mask=mask.to(cuda_dev))
        y.backward(gout)
        outs.append(y)
    assert rel_err(outs[0], fused_ref) <= FP32_TOL
    assert torch.equal(outs[0], outs[1])                          # recomputation reproduces the forward
    assert torch.equal(xs[0].grad, xs[1].grad)
    for (name, p), q in zip(mod.named_parameters(), plain.parameters()):
        assert (p.grad is None) == (q.grad is None), name
        if p.grad is not None:
            assert torch.equal(p.grad, q.grad), name
    _relation4_grads_are_zero(mod)


def test_graphed_typed_gat_encoder_step_equals_eager(cuda_dev):
    torch.manual_seed(3)
    n, e, f, h = 3000, 9000, 300, 64
    ei = synth.rmat_edges(n, e, seed=11).to(cuda_dev)
    enc = G.GraphEncoder(f, h, 96, dropout_rate=0.0, conv="gat", heads=8, gat_edge_types=True).to(cuda_dev)
    xs = [torch.randn(n, f, device=cuda_dev) for _ in range(3)]
    gy = torch.randn(n, 96, device=cuda_dev)
    step = G.GraphedEncoderStep(enc, xs[0], ei, autocast=True, x_requires_grad=True)
    assert step.edge_type is not None
    replayed = []
    for x in xs[1:]:
        y = step(x, gy).clone()
        grads = {k: p.grad.clone() for k, p in enc.named_parameters() if p.grad is not None}
        replayed.append((y, step.input_grad.clone(), grads))
    assert {f"gat{k}.{p}" for k in range(1, 5) for p in ("lin_edge.weight", "att_edge")} <= set(replayed[0][2])
    for x, (y, gx, grads) in zip(xs[1:], replayed):
        enc.zero_grad(set_to_none=True)
        xe = x.clone().requires_grad_(True)
        with torch.amp.autocast("cuda"):
            ye = enc.get_graph_embeddings(xe, ei)
        ye.backward(gy)
        assert torch.equal(y, ye)
        assert torch.equal(gx, xe.grad)
        for k, p in enc.named_parameters():
            if p.grad is not None:
                assert torch.equal(grads[k], p.grad), k
    _relation4_grads_are_zero(enc)
