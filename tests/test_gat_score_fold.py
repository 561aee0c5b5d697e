"""CPU, fp64: the GAT score folding behind GATConv's autocast path.  ``x @ gat_score_weight(W, att_src, att_dst).T``
must equal ``[z | (z*att_src).sum(-1) | (z*att_dst).sum(-1)]`` with ``z = x @ W.T``, and its gradients with respect
to x, W, att_src and att_dst must equal autograd of that unfused form."""
import pytest
import torch

from gmlm_b200.attn import gat_score_weight


@pytest.mark.parametrize("n,k,heads,c", [(37, 300, 8, 64), (5, 16, 3, 7), (1, 4, 1, 1)])
def test_folded_scores_equal_the_unfused_form(n, k, heads, c):
    gen = torch.Generator().manual_seed(n + k + heads + c)
    x = torch.randn(n, k, generator=gen, dtype=torch.float64)
    w = torch.randn(heads * c, k, generator=gen, dtype=torch.float64) / k ** 0.5
    att_s = torch.randn(1, heads, c, generator=gen, dtype=torch.float64)
    att_d = torch.randn(1, heads, c, generator=gen, dtype=torch.float64)
    gout = torch.randn(n, heads * c + 2 * heads, generator=gen, dtype=torch.float64)

    leaves = [t.clone().requires_grad_(True) for t in (x, w, att_s, att_d)]
    xf, wf, asf, adf = leaves
    y = xf @ gat_score_weight(wf, asf, adf).t()
    y.backward(gout)

    ref_leaves = [t.clone().requires_grad_(True) for t in (x, w, att_s, att_d)]
    xr, wr, asr, adr = ref_leaves
    z = xr @ wr.t()
    zv = z.view(n, heads, c)
    ref = torch.cat([z, (zv * asr).sum(-1), (zv * adr).sum(-1)], dim=1)
    ref.backward(gout)

    assert y.shape == (n, heads * c + 2 * heads)
    scale = float(ref.detach().abs().max())
    assert float((y - ref).abs().max()) <= 1e-12 * scale
    for got, want in zip(leaves, ref_leaves):
        assert float((got.grad - want.grad).abs().max()) <= 1e-12 * float(want.grad.abs().max())
