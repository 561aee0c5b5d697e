"""Graph ingest on the way INTO the hot path (SURVEY §8f row N3): the reference's ``.npz`` loader
(``load_npz_dataset``, ``/root/reference/main.py:780-820``), its 10 % edge dropout (``augment_graph``,
``main.py:832-837``) and the hand-off to the CSR build.

* ``load_npz_graph`` reads the same keys with the same dtypes and reproduces the seeded split of the reference
  function (``np.random.RandomState(seed).shuffle``) -- host logic, bit-identical (tests/test_ingest.py runs the
  reference's own function beside it).  It returns a plain namespace: the reference wraps the same tensors in a
  ``torch_geometric.data.Data``.
* ``edge_dropout_mask`` draws the keep mask exactly as ``augment_graph`` does (``torch.rand(E) > p`` on the CPU
  generator), so a seeded run keeps the same edges; ``augment_graph`` applies it the reference's way (a filtered
  ``edge_index``), while ``build_dropped_graph`` feeds the MASK to the CSR build (``RelGraph.build(keep_mask=...)``,
  ``gmlm_csr_build`` / ``gmlm_degree_i32_masked``): the edge typing sees the post-dropout degrees, as in the
  reference where the dropped ``edge_index`` replaces the original one, and no filtered edge list is materialised.
* ``save_rel_graph`` / ``load_rel_graph``: the built CSR pair as one ``.pt`` file, so that the sort of a 2e8-edge
  graph is paid once per dataset, not once per process.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib
from .graph import CSR, RelGraph, _ptr, _require_cuda, _stream


def load_npz_graph(npz_path: str, split_ratios: Optional[Tuple[float, float, float]] = None, seed: int = 42):
    """``load_npz_dataset`` (main.py:780-820) without the ``Data`` wrapper: returns (data, num_features, num_classes)
    with ``data.x`` float32 [N,F], ``data.edge_index`` int64 [2,E], ``data.y``, ``node_texts``, ``label_texts`` and the
    three boolean masks."""
    d = np.load(npz_path, allow_pickle=True)
    x = torch.tensor(d["node_features"], dtype=torch.float)
    edge_index = torch.tensor(d["edges"], dtype=torch.long)
    y = torch.tensor(d["node_labels"], dtype=torch.long)
    node_texts, label_texts = list(d["node_texts"]), list(d["label_texts"])
    num_nodes = x.size(0)
    if split_ratios is not None:
        train_ratio, val_ratio, _ = split_ratios
        idx = np.arange(num_nodes)
        np.random.RandomState(seed).shuffle(idx)
        n_train, n_val = int(train_ratio * num_nodes), int(val_ratio * num_nodes)
        masks = []
        for part in (idx[:n_train], idx[n_train:n_train + n_val], idx[n_train + n_val:]):
            m = torch.zeros(num_nodes, dtype=torch.bool)
            m[part] = True
            masks.append(m)
    else:
        masks = [torch.tensor(d[k], dtype=torch.bool) for k in ("train_masks", "val_masks", "test_masks")]
    data = SimpleNamespace(x=x, edge_index=edge_index, y=y, node_texts=node_texts, label_texts=label_texts,
                           train_mask=masks[0], val_mask=masks[1], test_mask=masks[2])
    return data, x.size(1), len(set(y.tolist()))


def edge_dropout_mask(num_edges: int, edge_dropout_p: float = 0.1, generator: Optional[torch.Generator] = None):
    """The keep mask of ``augment_graph`` (main.py:835): ``torch.rand(num_edges) > p`` on the CPU generator."""
    return torch.rand(num_edges, generator=generator) > edge_dropout_p


def augment_graph(data, edge_dropout_p: float = 0.1, generator: Optional[torch.Generator] = None):
    """Drop-in for ``augment_graph`` (main.py:832-837): replaces ``data.edge_index`` by the kept edges."""
    keep = edge_dropout_mask(data.edge_index.size(1), edge_dropout_p, generator)
    data.edge_index = data.edge_index[:, keep]
    return data


def build_dropped_graph(edge_index: torch.Tensor, keep_mask: torch.Tensor, num_nodes: int, num_relations: int = 5,
                        bounds=(2, 5, 10)) -> RelGraph:
    """Edge dropout + degree-bucket typing (main.py:253-267 on the dropped graph) + CSR build, with the mask fused
    into every kernel instead of a filtered ``edge_index``: equals
    ``RelGraph.build(ei[:, keep], edge_type_from_degree(ei[:, keep]), ...)`` array for array."""
    lib = _lib.load()
    _require_cuda(edge_index, "edge_index")
    dev = edge_index.device
    ei = edge_index.long()
    src = ei[0].contiguous()
    keep = keep_mask.to(dev)
    keep_u8 = keep.contiguous().view(torch.uint8) if keep.dtype == torch.bool else (keep != 0).view(torch.uint8)
    with torch.cuda.device(dev):
        deg = torch.empty(num_nodes, dtype=torch.int32, device=dev)
        _lib.check(lib.gmlm_degree_i32_masked(_ptr(src), _ptr(keep_u8), src.numel(), num_nodes, _ptr(deg), 0,
                                              _stream(dev)), "degree_masked")
    et = torch.ops.gmlm.edge_type_bucket(src, deg, list(bounds))         # types of dropped edges are never read
    return RelGraph.build(ei, et, num_nodes, num_relations, keep_mask=keep)


_CSR_FIELDS = ("rowptr", "col", "w", "perm", "hub_row", "hub_chunk_ptr", "chunk_beg", "chunk_end", "grp_row", "hub_col",
               "hub_w", "band_plan")


def save_rel_graph(graph: RelGraph, path: str) -> None:
    """The CSR pair (with its hub and group plans) as one file."""
    def pack(c: CSR):
        d = {k: (getattr(c, k).cpu() if getattr(c, k) is not None else None) for k in _CSR_FIELDS}
        d.update(num_rows=c.num_rows, hub_thresh=c.hub_thresh, n_hub=c.n_hub, n_chunks=c.n_chunks, quantum=c.quantum,
                 n_groups=c.n_groups)
        return d
    torch.save({"format": "gmlm_b200.RelGraph/1", "num_nodes": graph.num_nodes, "num_edges": graph.num_edges,
                "num_relations": graph.num_relations, "live_rels": list(graph.live_rels), "num_src": graph.num_src,
                "fwd": pack(graph.fwd), "bwd": pack(graph.bwd)}, path)


def load_rel_graph(path: str, device) -> RelGraph:
    blob = torch.load(path, map_location="cpu", weights_only=True)
    if blob.get("format") != "gmlm_b200.RelGraph/1":
        raise _lib.GmlmError(f"{path}: not a gmlm_b200 RelGraph file")
    dev = torch.device(device)
    if dev.type != "cuda":
        raise _lib.GmlmError("load_rel_graph: the graph lives on a CUDA device (no CPU path)")

    def unpack(d):
        kw = {k: (d[k].to(dev) if d.get(k) is not None else None) for k in _CSR_FIELDS}   # files without a band plan: none
        return CSR(num_rows=d["num_rows"], hub_thresh=d["hub_thresh"], n_hub=d["n_hub"], n_chunks=d["n_chunks"],
                   quantum=d["quantum"], n_groups=d["n_groups"], **kw)
    return RelGraph(num_nodes=blob["num_nodes"], num_edges=blob["num_edges"], num_relations=blob["num_relations"],
                    live_rels=list(blob["live_rels"]), fwd=unpack(blob["fwd"]), bwd=unpack(blob["bwd"]),
                    num_src=blob["num_src"])
