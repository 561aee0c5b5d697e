"""fp64-capable stock-torch restatement of upstream ``GATConv(edge_dim=D)`` and of the GAT encoder whose layers
attend over the degree-bucket edge types (test and measurement support).

``GATConvEdgeRef`` is ``oracle.GATConvRef`` (unchanged without ``edge_dim``) plus upstream's edge features, restated
literally as PyG 2.5/2.6 runs them, with no folding:
  * ``lin_edge = Linear(D, H*C, bias=False)`` and ``att_edge [1, H, C]``, both glorot;
  * ``remove_self_loops(edge_index, edge_attr)`` drops input self-loops with their attributes, then
    ``add_self_loops(..., fill_value="mean")`` appends one loop per node whose attribute is the mean of the
    attributes of the node's remaining in-edges (``edge_index[1] == i``), or 0 without any;
  * ``alpha_edge = (lin_edge(edge_attr).view(E, H, C) * att_edge).sum(-1)`` is added to ``a_src[j] + a_dst[i]``
    before the leaky ReLU; the softmax, ``+1e-16`` and attention dropout are the oracle's.

``TypedGATEncoderRef`` is ``GATEncoderRef`` with ``gat1..gat4 = GATConvEdgeRef(..., edge_dim=5)``, fed the one-hot of
the oracle's ``edge_type_bucket_ref`` (main.py:253-267).  Its submodule and parameter names equal those of
``gmlm_b200.GraphEncoder(conv="gat", gat_edge_types=True)``, so a state dict moves between the two.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import EncoderRef, GATConvRef
from oracle.pyg_ref import glorot_

from gat_encoder_ref import GATEncoderRef

NUM_RELATIONS = 5


def loop_fill_mean_ref(edge_index: torch.Tensor, edge_attr: torch.Tensor, num_nodes: int):
    """``remove_self_loops`` + ``add_self_loops(fill_value="mean")`` on ``(edge_index, edge_attr)``: the kept edges
    in input order, then loops 0..N-1 whose attribute is the scatter-mean over ``edge_index[1]`` of the kept ones."""
    keep = edge_index[0] != edge_index[1]
    edge_index, edge_attr = edge_index[:, keep], edge_attr[keep]
    summed = torch.zeros((num_nodes, edge_attr.size(1)), dtype=edge_attr.dtype,
                         device=edge_attr.device).index_add_(0, edge_index[1], edge_attr)
    cnt = torch.zeros((num_nodes,), dtype=edge_attr.dtype, device=edge_attr.device).index_add_(
        0, edge_index[1], torch.ones(edge_index.size(1), dtype=edge_attr.dtype, device=edge_attr.device))
    loop_attr = summed / cnt.clamp(min=1).unsqueeze(-1)
    loops = torch.arange(num_nodes, dtype=edge_index.dtype, device=edge_index.device)
    return torch.cat([edge_index, torch.stack([loops, loops])], dim=1), torch.cat([edge_attr, loop_attr], dim=0)


class GATConvEdgeRef(GATConvRef):
    def __init__(self, in_channels: int, out_channels: int, heads: int = 1, concat: bool = True,
                 negative_slope: float = 0.2, dropout: float = 0.0, edge_dim=None):
        super().__init__(in_channels, out_channels, heads=heads, concat=concat, negative_slope=negative_slope,
                         dropout=dropout)
        self.edge_dim = edge_dim
        if edge_dim is not None:
            self.lin_edge = nn.Linear(edge_dim, heads * out_channels, bias=False)
            self.att_edge = nn.Parameter(torch.empty(1, heads, out_channels))
            glorot_(self.lin_edge.weight)
            glorot_(self.att_edge)

    def forward(self, x: torch.Tensor, edge_index: torch.Tensor, edge_attr=None) -> torch.Tensor:
        if self.edge_dim is None or edge_attr is None:
            return super().forward(x, edge_index)
        n, hd, c = x.size(0), self.heads, self.out_channels
        z = self.lin(x).view(n, hd, c)
        a_src = (z * self.att_src).sum(-1)
        a_dst = (z * self.att_dst).sum(-1)
        if edge_attr.dim() == 1:
            edge_attr = edge_attr.view(-1, 1)
        ei, ea = loop_fill_mean_ref(edge_index.long(), edge_attr, n)
        src, dst = ei[0], ei[1]
        alpha_edge = (self.lin_edge(ea).view(-1, hd, c) * self.att_edge).sum(-1)
        e = F.leaky_relu(a_src[src] + a_dst[dst] + alpha_edge, self.negative_slope)        # [E', hd]
        emax = torch.full((n, hd), float("-inf"), dtype=e.dtype, device=e.device)
        emax = emax.scatter_reduce(0, dst.unsqueeze(-1).expand_as(e), e.detach(), reduce="amax", include_self=True)
        ex = (e - emax[dst]).exp()
        den = torch.zeros((n, hd), dtype=e.dtype, device=e.device).index_add_(0, dst, ex) + 1e-16
        alpha = ex / den[dst]
        alpha = F.dropout(alpha, p=self.dropout, training=self.training)
        out = torch.zeros((n, hd, c), dtype=z.dtype, device=z.device).index_add_(
            0, dst, alpha.unsqueeze(-1) * z.index_select(0, src))
        out = out.reshape(n, hd * c) if self.concat else out.mean(dim=1)
        return out + self.bias


class TypedGATEncoderRef(GATEncoderRef):
    def __init__(self, gnn_in_channels: int, hidden_channels: int, out_dim: int, heads: int = 8,
                 dropout_rate: float = 0.3, use_checkpoint: bool = True):
        super().__init__(gnn_in_channels, hidden_channels, out_dim, heads=heads, dropout_rate=dropout_rate,
                         use_checkpoint=use_checkpoint)
        h = hidden_channels
        dims = [gnn_in_channels, h, 2 * h, 4 * h, 8 * h]
        for k in range(4):
            setattr(self, f"gat{k+1}", GATConvEdgeRef(dims[k], dims[k + 1] // heads, heads=heads,
                                                      edge_dim=NUM_RELATIONS))

    def _block(self, k: int):
        conv, norm, drop = getattr(self, f"gat{k}"), getattr(self, f"gnorm{k}"), getattr(self, f"dropout{k}")

        def run(x, edge_index, edge_type):
            y = conv(x, edge_index, F.one_hot(edge_type.long(), NUM_RELATIONS).to(x.dtype))
            if y.size(0) > 1:
                y = norm(y)
            return drop(nn.functional.gelu(y))
        return run

    def forward(self, x_feat, edge_index, edge_type=None, return_layers: bool = False):
        # the oracle computes the degree-bucket types when none are given (main.py:253-267)
        return EncoderRef.forward(self, x_feat, edge_index, edge_type, return_layers=return_layers)
