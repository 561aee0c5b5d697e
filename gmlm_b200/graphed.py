"""CUDA-graphed encoder step for the small graphs (BASELINE configs[0..2]: Cornell-, Roman-empire-, Amazon-ratings-
shaped; SURVEY §7 step 9).

On these graphs one encoder forward+backward is ~140 kernels of a few microseconds to a millisecond each; the
reference's training loops (``/root/reference/main.py:439-454, 530-562``) call it once or twice per step on a static
graph with static shapes.  ``GraphedEncoderStep`` captures forward + backward once (the documented whole-network
capture pattern of ``torch.cuda.graphs``) and replays it: one graph launch per step instead of ~140 kernel launches
plus the Python/dispatcher time between them.  The C-ABI kernels launch on the capturing stream like any torch
operator; nothing on the path synchronises (the graph cache hits on tensor identity, tensor maps are cached by
address, which the graph's private memory pool keeps stable).

    step = GraphedEncoderStep(encoder, x, edge_index)          # captures
    y = step(x_new, grad_out)                                  # replays; parameter .grad tensors are refilled
"""
from __future__ import annotations

from typing import Optional

import torch

from .encoder import GraphEncoder, cached_edge_type


class GraphedEncoderStep:
    def __init__(self, encoder: GraphEncoder, x: torch.Tensor, edge_index: torch.Tensor,
                 edge_type: Optional[torch.Tensor] = None, autocast: bool = True, x_requires_grad: bool = False,
                 warmup: int = 3):
        if not x.is_cuda:
            raise RuntimeError("GraphedEncoderStep: CUDA tensors only (there is no CPU path)")
        self.encoder = encoder
        self.autocast = bool(autocast)
        n = x.size(0)
        self.edge_index = edge_index
        typed = getattr(encoder, "conv", "rgcn") == "rgcn" or getattr(encoder, "gat_edge_types", False)
        if edge_type is None and typed:
            edge_type = cached_edge_type(edge_index, n)           # GAT layers take none unless gat_edge_types
        self.edge_type = edge_type
        self.static_x = x.detach().clone().requires_grad_(x_requires_grad)
        side = torch.cuda.Stream(device=x.device)
        side.wait_stream(torch.cuda.current_stream(x.device))
        with torch.cuda.stream(side):                         # warm-up off the capture: builds the CSR, the plans,
            for _ in range(max(1, warmup)):                   # the tensor maps and the allocator's pools
                y = self._forward()
                y.backward(torch.ones_like(y))
                self._clear_grads()
        torch.cuda.current_stream(x.device).wait_stream(side)
        torch.cuda.synchronize(x.device)
        self.static_gy = torch.ones_like(y)
        del y
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.static_y = self._forward()
            self.static_y.backward(self.static_gy)            # parameter grads are allocated from the graph's pool:
        torch.cuda.synchronize(x.device)                      # every replay refills the same .grad tensors

    def _forward(self) -> torch.Tensor:
        with torch.amp.autocast("cuda", enabled=self.autocast):
            return self.encoder.get_graph_embeddings(self.static_x, self.edge_index, self.edge_type)

    def _clear_grads(self):
        self.encoder.zero_grad(set_to_none=True)
        self.static_x.grad = None

    def __call__(self, x: Optional[torch.Tensor] = None, grad_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Replay: ``x`` / ``grad_out`` are copied into the captured buffers (None = keep the previous contents);
        returns the captured output tensor; parameter gradients are in ``p.grad`` (overwritten, not accumulated)."""
        if x is not None:
            self.static_x.detach().copy_(x)
        if grad_out is not None:
            self.static_gy.copy_(grad_out)
        self.graph.replay()
        return self.static_y

    @property
    def input_grad(self) -> Optional[torch.Tensor]:
        return self.static_x.grad
