"""fp64-capable stock-torch restatement of the encoder body on GAT layers (test and measurement support).

``GATEncoderRef`` is ``oracle.EncoderRef`` with its four RGCN layers replaced by ``gat1..gat4 =
GATConvRef(dims[k], dims[k+1] // heads, heads)`` (concatenated heads, attention dropout 0, upstream's defaults).
Everything else is the oracle's: ``gnorm1..4``, ``dropout1..4``, ``residual_proj1..3``, ``multi_scale_fusion``,
the residual placement, the N > 1 GraphNorm gate and the dead third residual.  Submodule names equal those of
``gmlm_b200.GraphEncoder(conv="gat")``, so a state dict moves between the two.  GAT layers take no edge types.
"""
import torch.nn as nn

from oracle import EncoderRef, GATConvRef


class GATEncoderRef(EncoderRef):
    def __init__(self, gnn_in_channels: int, hidden_channels: int, out_dim: int, heads: int = 8,
                 dropout_rate: float = 0.3, use_checkpoint: bool = True):
        super().__init__(gnn_in_channels, hidden_channels, out_dim, dropout_rate=dropout_rate,
                         use_checkpoint=use_checkpoint)
        h = hidden_channels
        dims = [gnn_in_channels, h, 2 * h, 4 * h, 8 * h]
        for k in range(4):
            delattr(self, f"rgcn{k+1}")
            setattr(self, f"gat{k+1}", GATConvRef(dims[k], dims[k + 1] // heads, heads=heads))

    def _block(self, k: int):
        conv, norm, drop = getattr(self, f"gat{k}"), getattr(self, f"gnorm{k}"), getattr(self, f"dropout{k}")

        def run(x, edge_index, edge_type):             # as EncoderRef._block, conv without edge types
            y = conv(x, edge_index)
            if y.size(0) > 1:
                y = norm(y)
            return drop(nn.functional.gelu(y))
        return run

    def forward(self, x_feat, edge_index, edge_type=None, return_layers: bool = False):
        # a placeholder edge_type keeps the oracle from computing degree buckets GAT layers do not use
        return super().forward(x_feat, edge_index, edge_index.new_zeros(0) if edge_type is None else edge_type,
                               return_layers=return_layers)
