"""CPU, fp64: GATConv with edge features (upstream ``GATConv(edge_dim=D)``).

* a hand-derived known answer for the edge-aware oracle (``GATConvEdgeRef``) on three nodes, with an input self-loop
  (dropped with its attribute), a node without in-edges (its loop attribute is 0) and a duplicate edge;
* the fold behind ``GATConv``'s edge term: ``edge_attr @ gat_edge_weight(lin_edge.weight, att_edge).T`` equals the
  oracle's unfolded ``(lin_edge(edge_attr).view(E, H, C) * att_edge).sum(-1)``, values and gradients;
* the layer's and the encoder's parameter names and shapes, which state dicts depend on, and the argument checks
  that run before any device work."""
import math

import pytest
import torch

import gmlm_b200 as G
from gmlm_b200.attn import gat_edge_weight

from gat_edge_ref import GATConvEdgeRef, TypedGATEncoderRef

# ------------------------------------------------------------------------------------------------ known answer
# one head, one channel, 1-D edge_attr (D = 1); x = (0, 1, -1); lin = 1 (z = x); att_src = 1, att_dst = 0 (so the
# node part of the score of j -> i is x_j); lin_edge = 2, att_edge = 1 (alpha_edge = 2 * attr); slope .2; bias .25.
# Edges (src -> dst, attr):  0 -> 1 (.5),  0 -> 1 (-.5, a duplicate),  2 -> 1 (1),  1 -> 2 (.25),  2 -> 2 (7, a loop).
#   remove_self_loops drops 2 -> 2 and its 7; add_self_loops(fill_value="mean") gives each node's loop the mean
#   attribute of its remaining in-edges:  node 0: none -> 0;  node 1: (.5 - .5 + 1) / 3 = 1/3;  node 2: .25.
#   node 0: its loop only -> alpha = 1 -> x0 = 0
#   node 1: e(0->1) = leaky(0 + 2*.5) = 1,  e(0->1)' = leaky(0 - 1) = -.2,  e(2->1) = leaky(-1 + 2) = 1,
#           e(1->1) = leaky(1 + 2/3) = 5/3;   out = (e^1 * 0 + e^-.2 * 0 + e^1 * -1 + e^(5/3) * 1) / (sum of the four)
#   node 2: e(1->2) = leaky(1 + .5) = 1.5,  e(2->2) = leaky(-1 + .5) = .2 * -.5 = -.1
#           out = (e^1.5 * 1 + e^-.1 * -1) / (e^1.5 + e^-.1)
KA_X = [[0.0], [1.0], [-1.0]]
KA_EDGES = [[0, 0, 2, 1, 2], [1, 1, 1, 2, 2]]
KA_ATTR = [0.5, -0.5, 1.0, 0.25, 7.0]
_E = math.exp
KA_WANT = [[0.0 + 0.25],
           [(-_E(1.0) + _E(5.0 / 3.0)) / (_E(1.0) + _E(-0.2) + _E(1.0) + _E(5.0 / 3.0)) + 0.25],
           [(_E(1.5) - _E(-0.1)) / (_E(1.5) + _E(-0.1)) + 0.25]]


def ka_params():
    one = torch.ones(1, 1, 1, dtype=torch.float64)
    return {"lin.weight": torch.ones(1, 1, dtype=torch.float64), "att_src": one, "att_dst": torch.zeros_like(one),
            "lin_edge.weight": torch.full((1, 1), 2.0, dtype=torch.float64), "att_edge": one.clone(),
            "bias": torch.full((1,), 0.25, dtype=torch.float64)}


def test_oracle_gat_edge_attr_known_answer():
    ref = GATConvEdgeRef(1, 1, heads=1, edge_dim=1).double().eval()
    ref.load_state_dict(ka_params())
    out = ref(torch.tensor(KA_X, dtype=torch.float64), torch.tensor(KA_EDGES),
              torch.tensor(KA_ATTR, dtype=torch.float64))
    assert torch.allclose(out, torch.tensor(KA_WANT, dtype=torch.float64), rtol=1e-12, atol=1e-12), out
    # without edge_attr the oracle is upstream's layer without edge features
    plain = ref(torch.tensor(KA_X, dtype=torch.float64), torch.tensor(KA_EDGES))
    assert not torch.allclose(plain, out)


# ------------------------------------------------------------------------------------------------ the fold
@pytest.mark.parametrize("e,d,heads,c", [(37, 5, 8, 64), (11, 1, 3, 7), (4, 16, 2, 5), (1, 1, 1, 1)])
def test_folded_edge_scores_equal_the_unfolded_form(e, d, heads, c):
    gen = torch.Generator().manual_seed(e * 100 + d + heads + c)
    ea = torch.randn(e, d, generator=gen, dtype=torch.float64)
    w = torch.randn(heads * c, d, generator=gen, dtype=torch.float64) / d ** 0.5
    att = torch.randn(1, heads, c, generator=gen, dtype=torch.float64)
    gout = torch.randn(e, heads, generator=gen, dtype=torch.float64)

    leaves = [t.clone().requires_grad_(True) for t in (ea, w, att)]
    eaf, wf, attf = leaves
    y = eaf @ gat_edge_weight(wf, attf).t()
    y.backward(gout)

    ref = GATConvEdgeRef(3, c, heads=heads, edge_dim=d).double()
    ref_leaves = [ea.clone().requires_grad_(True)]
    with torch.no_grad():
        ref.lin_edge.weight.copy_(w)
        ref.att_edge.copy_(att)
    want = (ref.lin_edge(ref_leaves[0]).view(e, heads, c) * ref.att_edge).sum(-1)
    want.backward(gout)

    assert y.shape == (e, heads)
    assert float((y - want).detach().abs().max()) <= 1e-12 * float(want.detach().abs().max())
    for got, exp in zip(leaves, [ref_leaves[0].grad, ref.lin_edge.weight.grad, ref.att_edge.grad]):
        assert float((got.grad - exp).abs().max()) <= 1e-12 * float(exp.abs().max())


# ------------------------------------------------------------------------------------------------ names and checks
def test_gat_conv_edge_parameters_match_upstream_names():
    mod = G.GATConv(12, 4, heads=3, edge_dim=5)
    sd = mod.state_dict()
    assert sd["lin_edge.weight"].shape == (12, 5) and sd["att_edge"].shape == (1, 3, 4)
    ref = GATConvEdgeRef(12, 4, heads=3, edge_dim=5)
    assert {k: v.shape for k, v in ref.state_dict().items()} == {k: v.shape for k, v in sd.items()}
    assert mod.load_state_dict(ref.state_dict()) is not None
    plain = G.GATConv(12, 4, heads=3)                          # no edge_dim: today's parameters, nothing more
    assert set(plain.state_dict()) == {"lin.weight", "att_src", "att_dst", "bias"}
    assert plain.lin_edge is None and plain.att_edge is None


def test_gat_conv_rejects_other_fill_values():
    for fill in ("add", 0.0, "max"):
        with pytest.raises(NotImplementedError, match="fill_value"):
            G.GATConv(4, 4, edge_dim=2, fill_value=fill)


def test_gat_conv_positional_arguments_are_not_misrouted():
    """PyG's order is forward(x, edge_index, edge_attr); the dropout seed goes by keyword.  An int where edge_attr
    goes (an old positional seed) and a tensor or a non-int where the seed goes raise instead of being dropped."""
    mod = G.GATConv(4, 2, heads=2, edge_dim=3, dropout=0.5)
    x, ei = torch.randn(3, 4), torch.tensor([[0, 1], [1, 2]])
    with pytest.raises(TypeError, match="edge_attr must be a tensor"):
        mod(x, ei, 1234)
    with pytest.raises(TypeError, match="dropout_seed must be an int"):
        mod(x, ei, None, torch.randn(2, 3))
    with pytest.raises(TypeError, match="dropout_seed must be an int"):
        mod(x, ei, dropout_seed=torch.tensor(7))
    with pytest.raises(TypeError, match="dropout_seed must be an int"):
        mod(x, ei, dropout_seed=1.5)
    with pytest.raises(TypeError, match="dropout_seed must be an int"):
        mod(x, ei, dropout_seed=True)


def test_typed_gat_encoder_state_dict_keys():
    mod = G.GraphEncoder(64, 16, 32, conv="gat", heads=4, gat_edge_types=True)
    ref = TypedGATEncoderRef(64, 16, 32, heads=4, dropout_rate=0.0)
    sd, sd_ref = mod.state_dict(), ref.state_dict()
    assert set(sd) == set(sd_ref) | {"gnn_mask_token_embed"}
    for k, v in sd_ref.items():
        assert sd[k].shape == v.shape, k
    dims = [64, 16, 32, 64, 128]
    for k in range(1, 5):
        assert sd[f"gat{k}.lin_edge.weight"].shape == (dims[k], 5)
        assert sd[f"gat{k}.att_edge"].shape == (1, 4, dims[k] // 4)
    assert not any("edge" in k for k in G.GraphEncoder(64, 16, 32, conv="gat", heads=4).state_dict())
    with pytest.raises(ValueError, match="gat_edge_types"):
        G.GraphEncoder(64, 16, 32, gat_edge_types=True)         # the RGCN encoder has its own relations
