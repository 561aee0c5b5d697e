"""GPU: the GMLM encoder on GAT edge-softmax layers (BASELINE configs[2]).

* the fused GAT kernels on rows wider than one warp covers (head groups over grid.y), fp32 and bf16 z, with hub
  chunks: forward and dz / da_src / da_dst against autograd of the fp64 two-pass softmax, run-to-run bit equality,
  and attention dropout that applies exactly ``gat_dropout_mask``;
* ``GATConv`` under autocast (one tcgen05 GEMM writes [z | a_src | a_dst]) against ``GATConvRef`` in fp64;
* ``GraphEncoder(conv="gat")`` against ``GATEncoderRef`` (oracle.EncoderRef on GATConvRef layers): fp32, autocast
  at hidden_channels = 512 (layers up to 4096 features), soft masking with checkpointing, and ``GraphedEncoderStep``
  replay."""
import copy

import pytest
import torch
import torch.nn.functional as F

import gmlm_b200 as G
from gmlm_b200 import _lib, synth
from gmlm_b200.attn import LoopGraph, gat_aggregate, gat_dropout_mask, gat_score_weight
from gmlm_b200.ops import linear_nt
from oracle import GATConvRef, soft_masking_ref

from conftest import rel_err
from gat_encoder_ref import GATEncoderRef

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
BF16_TOL = 2e-2


def _loopy_hub_graph(n, e, seed):
    """uniform edges with duplicates and self-loops, plus a star into node 7 so that hub_thresh = 32 cuts rows"""
    ei = synth.uniform_edges(n, e, seed=seed)
    ei[1, : e // 20] = ei[0, : e // 20]                       # self-loops (upstream removes then re-adds them)
    ei[:, e // 20: e // 10] = ei[:, : e // 20]                # duplicate edges
    star = torch.stack([torch.arange(n), torch.full((n,), 7)])
    return torch.cat([ei, star, star[:, :40]], dim=1)


def _reference(graph, z, a_s, a_d, keep=None, p=0.0, slope=0.2):
    """fp64 two-pass edge softmax in forward-CSR order, differentiable in z, a_src, a_dst"""
    rowptr, col = graph.fwd.rowptr.cpu().long(), graph.fwd.col.cpu().long()
    n, heads = a_d.shape
    c = z.size(1) // heads
    dst = torch.repeat_interleave(torch.arange(n), rowptr[1:] - rowptr[:-1])
    sc = F.leaky_relu(a_s[col] + a_d[dst], slope)
    emax = torch.full((n, heads), float("-inf"), dtype=torch.float64).scatter_reduce(
        0, dst.unsqueeze(-1).expand_as(sc), sc.detach(), reduce="amax", include_self=True)
    ex = (sc - emax[dst]).exp()
    alpha = ex / (torch.zeros((n, heads), dtype=torch.float64).index_add_(0, dst, ex) + 1e-16)[dst]
    if keep is not None:
        alpha = alpha * keep.cpu().double() / (1.0 - p)
    out = torch.zeros((n, heads, c), dtype=torch.float64).index_add_(0, dst, alpha.unsqueeze(-1) * z.view(n, heads, c)[col])
    return out.view(n, heads * c)


WIDE = [(8, 128), (8, 130), (8, 256), (8, 512), (3, 520)]


@pytest.fixture(scope="module")
def hub_graph(cuda_dev):
    n = 300
    ei = _loopy_hub_graph(n, 1500, seed=21).to(cuda_dev)
    graph = LoopGraph.build(ei, n, hub_thresh=32)
    assert graph.fwd.n_hub >= 1 and graph.fwd.n_chunks > graph.fwd.n_hub
    return n, graph


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("heads,c", WIDE)
def test_wide_rows_match_fp64_softmax(cuda_dev, hub_graph, heads, c, dtype):
    n, graph = hub_graph
    gen = torch.Generator().manual_seed(heads * 1000 + c)
    z = torch.randn(n, heads * c, generator=gen).to(dtype)
    a_s = torch.randn(n, heads, generator=gen) * 2
    a_d = torch.randn(n, heads, generator=gen) * 2
    gout = torch.randn(n, heads * c, generator=gen).to(dtype)

    zg = z.to(cuda_dev).requires_grad_(True)
    asg, adg = a_s.to(cuda_dev).requires_grad_(True), a_d.to(cuda_dev).requires_grad_(True)
    out = gat_aggregate(zg, asg, adg, graph)
    assert out.dtype == dtype
    out.backward(gout.to(cuda_dev))

    z64 = z.double().requires_grad_(True)
    as64, ad64 = a_s.double().requires_grad_(True), a_d.double().requires_grad_(True)
    ref = _reference(graph, z64, as64, ad64)
    ref.backward(gout.double())
    tol, gtol = (FP32_TOL, 2e-5) if dtype == torch.float32 else (BF16_TOL, BF16_TOL)
    assert rel_err(out, ref) <= tol
    assert rel_err(zg.grad, z64.grad) <= gtol
    assert rel_err(asg.grad, as64.grad) <= gtol and rel_err(adg.grad, ad64.grad) <= gtol

    # no atomics: a second run is bit-identical, forward and backward
    zg2 = zg.detach().clone().requires_grad_(True)
    as2, ad2 = asg.detach().clone().requires_grad_(True), adg.detach().clone().requires_grad_(True)
    out2 = gat_aggregate(zg2, as2, ad2, graph)
    out2.backward(gout.to(cuda_dev))
    assert torch.equal(out, out2)
    assert torch.equal(zg.grad, zg2.grad) and torch.equal(asg.grad, as2.grad) and torch.equal(adg.grad, ad2.grad)


@pytest.mark.parametrize("heads,c", WIDE)
def test_wide_rows_apply_the_hash_dropout_mask(cuda_dev, hub_graph, heads, c):
    """The head groups keep the global head index and H in the hash (seed, csr_pos * H + head)."""
    n, graph = hub_graph
    p, seed = 0.5, 987654321
    gen = torch.Generator().manual_seed(c)
    z = torch.randn(n, heads * c, generator=gen)
    a_s, a_d = torch.randn(n, heads, generator=gen), torch.randn(n, heads, generator=gen)
    keep = gat_dropout_mask(seed, graph.fwd.nnz, heads, p, cuda_dev)
    assert abs(float(keep.float().mean()) - (1 - p)) < 0.05
    zg = z.to(cuda_dev).requires_grad_(True)
    out = gat_aggregate(zg, a_s.to(cuda_dev), a_d.to(cuda_dev), graph, 0.2, p, seed)
    z64 = z.double().requires_grad_(True)
    ref = _reference(graph, z64, a_s.double(), a_d.double(), keep=keep, p=p)
    assert rel_err(out, ref) <= FP32_TOL
    assert torch.equal(out, gat_aggregate(zg.detach(), a_s.to(cuda_dev), a_d.to(cuda_dev), graph, 0.2, p, seed))
    gout = torch.randn(n, heads * c, generator=gen)
    out.backward(gout.to(cuda_dev))
    ref.backward(gout.double())
    assert rel_err(zg.grad, z64.grad) <= 2e-5


def test_a_head_wider_than_the_kernel_raises(cuda_dev, hub_graph):
    n, graph = hub_graph
    z = torch.randn(n, 2 * 1028, device=cuda_dev)
    a = torch.randn(n, 2, device=cuda_dev)
    with pytest.raises(_lib.GmlmError, match="one head of head_dim = 1028"):
        gat_aggregate(z, a, a, graph)


# ------------------------------------------------------------------------------------------- GATConv under autocast
@pytest.mark.parametrize("heads,c", [(8, 64), (8, 512)])
def test_gat_conv_autocast_matches_oracle(cuda_dev, heads, c):
    """Output at the layer-level autocast gate 2e-3.  The gradients of a GAT layer are far more sensitive to the
    16-bit rounding of the projection's operands than its output: d_score = alpha (d_alpha - t) cancels wherever
    one edge dominates the softmax, so a 5e-4 relative change of z moves dx by ~1e-2 of its maximum.  The
    gradient gates are therefore max(layer gate, 3x the error of the fp64 oracle fed the same fp16-rounded x and
    W), as the encoder tests gate gradients against the fp32 oracle's own error."""
    torch.manual_seed(13)
    n, e, fi = 700, 6000, 300
    ei = _loopy_hub_graph(n, e, seed=c)
    ref = GATConvRef(fi, c, heads=heads).double()
    with torch.no_grad():
        ref.bias.uniform_(-0.1, 0.1)
    mod = G.GATConv(fi, c, heads=heads)
    mod.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    mod = mod.to(cuda_dev)
    x, gout = torch.randn(n, fi), torch.randn(n, heads * c)
    x64 = x.double().requires_grad_(True)
    y_ref = ref(x64, ei)
    y_ref.backward(gout.double())
    ref16 = copy.deepcopy(ref)                                    # the same oracle on fp16-rounded operands
    with torch.no_grad():
        ref16.lin.weight.copy_(ref.lin.weight.half().double())
    ref16.zero_grad()
    x16 = x.half().double().requires_grad_(True)
    ref16(x16, ei).backward(gout.double())
    xg = x.to(cuda_dev).requires_grad_(True)
    with torch.amp.autocast("cuda"):
        y = mod(xg, ei.to(cuda_dev))
    assert y.dtype == torch.float32
    y.backward(gout.to(cuda_dev))
    assert rel_err(y, y_ref) <= 2e-3
    noise = rel_err(x16.grad, x64.grad)
    assert rel_err(xg.grad, x64.grad) <= max(2e-3, 3.0 * noise), noise
    for name in ("lin.weight", "att_src", "att_dst", "bias"):
        got = dict(mod.named_parameters())[name].grad
        want, want16 = dict(ref.named_parameters())[name].grad, dict(ref16.named_parameters())[name].grad
        noise = rel_err(want16, want, floor=1e-2)
        assert rel_err(got, want, floor=1e-2) <= max(5e-3, 3.0 * noise), (name, noise)

    # the fused score columns of the same GEMM agree with the scores computed from its z columns
    with torch.no_grad():
        w_ext = gat_score_weight(mod.lin.weight, mod.att_src, mod.att_dst)
        yy = linear_nt(xg.detach(), w_ext, out_dtype=torch.float32, op_dtype=torch.float16).double()
    hc = heads * c
    zv = yy[:, :hc].view(n, heads, c)
    assert rel_err(yy[:, hc:hc + heads], (zv * mod.att_src.detach().double()).sum(-1)) <= 2e-3
    assert rel_err(yy[:, hc + heads:hc + 2 * heads], (zv * mod.att_dst.detach().double()).sum(-1)) <= 2e-3


# ------------------------------------------------------------------------------------------------ the GAT encoder
def _gat_encoder_pair(fin, hidden, out_dim, heads, use_checkpoint=False):
    torch.manual_seed(5)
    ref = GATEncoderRef(fin, hidden, out_dim, heads=heads, dropout_rate=0.0, use_checkpoint=False).double()
    with torch.no_grad():
        for k in range(1, 5):
            getattr(ref, f"gnorm{k}").mean_scale.uniform_(0.5, 1.0)
            getattr(ref, f"gat{k}").bias.uniform_(-0.1, 0.1)
    mod = G.GraphEncoder(fin, hidden, out_dim, dropout_rate=0.0, conv="gat", heads=heads,
                         use_checkpoint=use_checkpoint)
    keys = set(mod.state_dict())
    assert keys == set(ref.state_dict()) | {"gnn_mask_token_embed"}
    want = {f"gat{k}.{p}" for k in range(1, 5) for p in ("lin.weight", "att_src", "att_dst", "bias")}
    assert want <= keys and not any(k.startswith("rgcn") for k in keys)
    missing, unexpected = mod.load_state_dict({k: v.float() for k, v in ref.state_dict().items()}, strict=False)
    assert unexpected == [] and missing == ["gnn_mask_token_embed"]
    return ref, mod


def test_gat_encoder_constructor_checks():
    with pytest.raises(ValueError):
        G.GraphEncoder(300, 20, 32, conv="gat", heads=8)          # 8 does not divide 20
    with pytest.raises(NotImplementedError):
        G.GraphEncoder(300, 64, 32, conv="gat", heads=8, act_dtype=torch.bfloat16)
    enc = G.GraphEncoder(300, 64, 32)                             # the default stays RGCN
    assert any(k.startswith("rgcn1.") for k in enc.state_dict())


@pytest.mark.parametrize("n,e,fin,hidden,heads", [(183, 300, 64, 16, 4), (2000, 9000, 300, 16, 8)])
def test_gat_encoder_matches_oracle_fp32(cuda_dev, n, e, fin, hidden, heads):
    ref, mod = _gat_encoder_pair(fin, hidden, 48, heads)
    mod = mod.to(cuda_dev)
    ei = _loopy_hub_graph(n, e, seed=n + 3)
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
        noise = rel_err(sd32[name].grad, sd_ref[name].grad)
        assert rel_err(p.grad, sd_ref[name].grad) <= max(2e-5, 3.0 * noise), (name, noise)


def test_gat_encoder_autocast_at_amazon_ratings_scale(cuda_dev):
    """1/10-scale Amazon-ratings-shaped graph at hidden_channels = 512: the GAT layers reach 2048 and 4096 features
    (8 heads of 256 and 512), past what one warp covers."""
    n, e, fin, hidden = 2449, 9305, 300, 512
    ref, mod = _gat_encoder_pair(fin, hidden, 768, 8)
    mod = mod.to(cuda_dev)
    ref = ref.to(cuda_dev)                                        # fp64 reference on the GPU (4096-wide layers)
    ei = _loopy_hub_graph(n, e, seed=17).to(cuda_dev)
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


def test_gat_encoder_soft_mask_with_checkpointing(cuda_dev):
    n, e, fin, hidden, heads = 600, 3000, 64, 16, 4
    ref, mod = _gat_encoder_pair(fin, hidden, 32, heads, use_checkpoint=True)
    mod = mod.to(cuda_dev)
    plain = copy.deepcopy(mod)
    plain.use_checkpoint = False
    ei = _loopy_hub_graph(n, e, seed=77).to(cuda_dev)
    gen = torch.Generator().manual_seed(8)
    x = torch.randn(n, fin, generator=gen)
    mask = torch.rand(n, generator=gen) < 0.3
    tok = mod.gnn_mask_token_embed.detach().cpu()
    fused_ref = ref(soft_masking_ref(x.double(), mask, tok.double()), ei.cpu())
    gout = torch.randn(n, 32, generator=gen).to(cuda_dev)
    xs = [x.to(cuda_dev).requires_grad_(True) for _ in range(2)]
    outs = []
    for m, xg in zip((mod, plain), xs):
        y = m(xg, ei, edge_type=torch.zeros(1), gnn_perturb_mask=mask.to(cuda_dev))   # edge_type is ignored
        y.backward(gout)
        outs.append(y)
    assert rel_err(outs[0], fused_ref) <= FP32_TOL
    assert torch.equal(outs[0], outs[1])                          # recomputation reproduces the forward
    assert torch.equal(xs[0].grad, xs[1].grad)
    assert mod.gnn_mask_token_embed.grad is not None and bool(torch.isfinite(mod.gnn_mask_token_embed.grad).all())
    for (name, p), q in zip(mod.named_parameters(), plain.parameters()):
        assert (p.grad is None) == (q.grad is None), name
        if p.grad is not None:
            assert torch.equal(p.grad, q.grad), name


def test_graphed_gat_encoder_step_equals_eager(cuda_dev):
    torch.manual_seed(3)
    n, e, f, h = 3000, 9000, 300, 64
    ei = synth.rmat_edges(n, e, seed=11).to(cuda_dev)
    enc = G.GraphEncoder(f, h, 96, dropout_rate=0.0, conv="gat", heads=8).to(cuda_dev)
    xs = [torch.randn(n, f, device=cuda_dev) for _ in range(3)]
    gy = torch.randn(n, 96, device=cuda_dev)
    step = G.GraphedEncoderStep(enc, xs[0], ei, autocast=True, x_requires_grad=True)
    assert step.edge_type is None
    replayed = []
    for x in xs[1:]:
        y = step(x, gy).clone()
        grads = {k: p.grad.clone() for k, p in enc.named_parameters() if p.grad is not None}
        replayed.append((y, step.input_grad.clone(), grads))
    assert len(replayed[0][2]) >= 40
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
