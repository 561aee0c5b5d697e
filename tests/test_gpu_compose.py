"""Basis composition (SURVEY §8a row A4: [PyG] RGCNConv.forward ``weight = comp @ weight.view(B, -1)``, modules built
main.py:189-201) against an fp64 restatement: forward in both layouts and all three operand types, backward
(basis and coefficient gradients) against autograd, and the layer through the kernel against the oracle."""
import pytest
import torch

from gmlm_b200.ops import basis_compose, basis_compose_bwd

from conftest import rel_err

pytestmark = pytest.mark.gpu


def _params(nb, r, fi, fo, seed, dev):
    g = torch.Generator().manual_seed(seed)
    weight = torch.randn(nb, fi, fo, generator=g).to(dev)
    comp = torch.randn(r, nb, generator=g).to(dev)
    root = torch.randn(fi, fo, generator=g).to(dev)
    return weight, comp, root


@pytest.mark.parametrize("op,tol", [(torch.float32, 2e-6), (torch.bfloat16, 8e-3), (torch.float16, 1e-3)])
@pytest.mark.parametrize("fi,fo", [(64, 64), (300, 512), (256, 64), (33, 20), (1703, 512), (100, 7)])
@pytest.mark.parametrize("live", [(0, 1, 2, 3), (1, 3), (4,)])
@pytest.mark.parametrize("layout", ["agg", "tf"])
def test_compose_forward_layouts(cuda_dev, op, tol, fi, fo, live, layout):
    weight, comp, root = _params(30, 5, fi, fo, fi * fo, cuda_dev)
    wn, wt = basis_compose(weight, comp, root, live, op, layout)
    w = (comp.double()[list(live)] @ weight.double().view(30, -1)).view(len(live), fi, fo)
    slabs = torch.cat([w, root.double()[None]], dim=0)                       # [S+1, Fi, Fo]
    ref_n = slabs.reshape(-1, fo) if layout == "agg" else slabs.permute(1, 0, 2).reshape(fi, -1)
    assert wn.shape == ref_n.shape and wt.shape == ref_n.t().shape and wn.dtype == op and wt.dtype == op
    assert rel_err(wn, ref_n) <= tol
    assert torch.equal(wt, wn.t())                                           # same rounding in both layouts
    es = wn.element_size()
    assert (wn.stride(0) * es) % 16 == 0 and (wt.stride(0) * es) % 16 == 0   # TMA-readable pitches


def test_compose_forward_without_bases_or_root(cuda_dev):
    weight, _, root = _params(5, 5, 48, 40, 3, cuda_dev)
    wn, wt = basis_compose(weight, None, None, (0, 2, 3), torch.float32, "agg")
    assert torch.equal(wn, weight[[0, 2, 3]].reshape(-1, 40)) and torch.equal(wt, wn.t())


@pytest.mark.parametrize("fi,fo", [(64, 64), (300, 512), (257, 36), (2048, 256), (100, 7), (33, 22)])
@pytest.mark.parametrize("live", [(0, 1, 2, 3), (2,)])
@pytest.mark.parametrize("layout", ["agg", "tf"])
def test_compose_backward_matches_autograd(cuda_dev, fi, fo, live, layout):
    nb, r = 30, 5
    weight, comp, _ = _params(nb, r, fi, fo, fi + fo, cuda_dev)
    S = len(live)
    g = torch.Generator().manual_seed(7)
    dws = torch.randn(S, fi, fo, generator=g).to(cuda_dev)                   # gradient of the composed weights
    w64 = weight.double().requires_grad_(True)
    c64 = comp.double().requires_grad_(True)
    w = (c64[list(live)] @ w64.view(nb, -1)).view(S, fi, fo)
    (w * dws.double()).sum().backward()
    if layout == "agg":
        dw, ss, rs = dws.contiguous(), fi * fo, fo
    else:                                                                    # [Fi, (S+1)*Fo]: slabs side by side
        dw = torch.cat([dws.permute(1, 0, 2).reshape(fi, S * fo), torch.zeros(fi, fo, device=cuda_dev)], dim=1).contiguous()
        ss, rs = fo, (S + 1) * fo
    dweight, dcomp = basis_compose_bwd(weight, comp, dw, ss, rs, live)
    assert rel_err(dweight, w64.grad) <= 2e-6
    assert rel_err(dcomp, c64.grad) <= 2e-5
    dead = [k for k in range(r) if k not in live]
    assert torch.count_nonzero(dcomp[dead]) == 0                             # relations without edges: exact zeros
    again = basis_compose_bwd(weight, comp, dw, ss, rs, live)
    assert torch.equal(again[0], dweight) and torch.equal(again[1], dcomp)   # deterministic


@pytest.mark.parametrize("autocast", [False, True])
@pytest.mark.parametrize("fi,fo", [(300, 512), (64, 128)])
def test_rgcn_conv_fp32_and_autocast_through_the_composition_kernel(cuda_dev, autocast, fi, fo):
    """RGCNConv with fp32 activations (the reference's eval mode, main.py:603) and under torch.amp.autocast (its
    training mode, main.py:446): forward and every parameter gradient against the fp64 oracle."""
    import gmlm_b200 as G
    from gmlm_b200 import synth
    from oracle import RGCNConvRef, edge_type_bucket_ref
    n, e = 2000, 9000
    torch.manual_seed(1)
    ei = synth.rmat_edges(n, e, seed=5)
    et = edge_type_bucket_ref(ei, n)
    ref = RGCNConvRef(fi, fo, 5, 30).double()
    with torch.no_grad():
        ref.bias.uniform_(-0.1, 0.1)
    x = torch.randn(n, fi)
    gout = torch.randn(n, fo)
    x64 = x.double().requires_grad_(True)
    y_ref = ref(x64, ei, et)
    y_ref.backward(gout.double())
    mod = G.RGCNConv(fi, fo, 5, 30)
    mod.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    mod = mod.to(cuda_dev)
    xg = x.to(cuda_dev).requires_grad_(True)
    with torch.amp.autocast("cuda", enabled=autocast):
        y = mod(xg, ei.to(cuda_dev), et.to(cuda_dev))
    assert y.dtype == torch.float32
    y.backward(gout.to(cuda_dev))
    tol = 2e-3 if autocast else 1e-5                                          # fp16 operands vs fp32
    assert rel_err(y, y_ref) <= tol
    assert rel_err(xg.grad, x64.grad) <= tol
    for name in ("weight", "comp", "root", "bias"):
        assert rel_err(getattr(mod, name).grad, getattr(ref, name).grad) <= (5e-3 if autocast else 2e-5), name
