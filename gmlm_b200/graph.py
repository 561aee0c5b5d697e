"""Graph structure cache: the (dst,rel)-keyed CSR that replaces the per-call, per-relation
boolean-mask compaction of upstream ``RGCNConv.forward`` (SURVEY §8a row A3; call sites
``/root/reference/main.py:272,285,298,308``), its transpose for the backward gather (A14), and
the hub plan that keeps power-law rows balanced and deterministic.

Everything is built by the CUDA library (``csr_build`` / ``csr_transpose`` / ``hub_*`` in
include/gmlm_b200.h); this module only owns the tensors and the cache.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from collections import OrderedDict
from dataclasses import dataclass, field
from typing import List, Optional

import torch

from . import _lib

DEFAULT_HUB_THRESH = int(os.environ.get("GMLM_HUB_THRESH", "256"))
DEFAULT_QUANTUM = int(os.environ.get("GMLM_GROUP_QUANTUM", "512"))   # 0 = uniform 32-row groups
# Band-ordered hub plan (gmlm_hub_band_sort), keyed on the use rank of the gathered rows: a band is the next
# 2^HUB_BAND_SHIFT rows by use, 32 MB of 512-byte rows.  Of 2^16 / 2^17 / 2^18 rows, 2^16 gave the fastest hub
# kernels on the C5 and C4 graphs in both directions (DESIGN §4.1, profiles/r7_time_hub_chunks.jsonl).  A band
# boundary splits a chunk only when both pieces keep HUB_BAND_MIN_RUN edges: shorter pieces cost a partial row
# written and read for few gathered rows.
HUB_BAND_SHIFT = 16
HUB_BAND_MIN_RUN = 32


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(t.data_ptr()) if t is not None and t.numel() > 0 else C.c_void_p(0)


def _stream(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _require_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise _lib.GmlmError(
            f"{name} must be a CUDA tensor: gmlm_b200 runs only on the GPU (no CPU fallback); got device {t.device}")


@dataclass
class CSR:
    """One direction of the graph in CSR form plus its hub plan."""
    rowptr: torch.Tensor                       # int32 [num_rows+1]
    col: torch.Tensor                          # int32 [nnz]  (gather row of each edge)
    num_rows: int
    w: Optional[torch.Tensor] = None           # float32 [nnz] per-edge weight (weighted mode)
    perm: Optional[torch.Tensor] = None        # int32 [nnz] original edge position
    hub_thresh: int = DEFAULT_HUB_THRESH
    n_hub: int = 0
    n_chunks: int = 0
    hub_row: Optional[torch.Tensor] = None
    hub_chunk_ptr: Optional[torch.Tensor] = None
    chunk_beg: Optional[torch.Tensor] = None
    chunk_end: Optional[torch.Tensor] = None
    hub_col: Optional[torch.Tensor] = None     # int32 [hub edges] col of the hub rows, each row sorted by band key
    hub_w: Optional[torch.Tensor] = None       # float32 [hub edges] w in the same order (weighted CSRs)
    band_plan: Optional[torch.Tensor] = None   # int32 [band_chunk_ptr | cut | chunk_order] (include/gmlm_b200.h)
    quantum: int = 0                           # cost-balanced group plan (0 = uniform groups)
    n_groups: int = 0
    grp_row: Optional[torch.Tensor] = None     # int32 [n_groups+1]

    @property
    def nnz(self) -> int:
        return int(self.col.numel())

    def plan_groups(self, quantum: Optional[int] = None):
        """Cut the rows into groups of about ``quantum`` units of work (edges + rows)."""
        lib = _lib.load()
        if quantum is None:
            # DEFAULT_QUANTUM units per group on big graphs; small graphs (the reference's own
            # datasets) get smaller groups so that there are >= ~32 groups per SM to hide latency
            # (measured on the Roman-empire shape: 105 us at 512 vs 45 us at 32)
            q = DEFAULT_QUANTUM
            if q > 0:
                sms = torch.cuda.get_device_properties(self.rowptr.device).multi_processor_count
                q = max(32, min(q, (self.num_rows + self.nnz) // (sms * 32)))
        else:
            q = int(quantum)
        self.quantum = q
        if q <= 0 or self.num_rows == 0:
            self.n_groups, self.grp_row = 0, None
            return self
        dev = self.rowptr.device
        with torch.cuda.device(dev):
            self.n_groups = int(lib.gmlm_group_plan_size(self.num_rows, self.nnz, q))
            self.grp_row = torch.empty(self.n_groups + 1, dtype=torch.int32, device=dev)
            _lib.check(lib.gmlm_group_plan(_ptr(self.rowptr), self.num_rows, self.nnz, q, _ptr(self.grp_row),
                                           _stream(dev)), "group_plan")
        return self

    def plan_hubs(self, thresh: Optional[int] = None):
        """Split rows longer than ``thresh`` into fixed chunks (deterministic two-stage reduce)."""
        lib = _lib.load()
        self.hub_thresh = int(thresh if thresh is not None else self.hub_thresh)
        dev = self.rowptr.device
        with torch.cuda.device(dev):
            ws_bytes = lib.gmlm_csr_workspace_bytes(max(self.nnz, 1), self.num_rows)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            counts = (C.c_int64 * 2)()
            _lib.check(lib.gmlm_hub_count(_ptr(self.rowptr), self.num_rows, self.hub_thresh, counts, _ptr(ws),
                                          ws_bytes, _stream(dev)), "hub_count")
            self.n_hub, self.n_chunks = int(counts[0]), int(counts[1])
            if self.n_hub:
                self.hub_row = torch.empty(self.n_hub, dtype=torch.int32, device=dev)
                self.hub_chunk_ptr = torch.empty(self.n_hub + 1, dtype=torch.int32, device=dev)
                self.chunk_beg = torch.empty(self.n_chunks, dtype=torch.int32, device=dev)
                self.chunk_end = torch.empty(self.n_chunks, dtype=torch.int32, device=dev)
                _lib.check(lib.gmlm_hub_fill(_ptr(self.rowptr), self.num_rows, self.hub_thresh, self.n_hub,
                                             self.n_chunks, _ptr(self.hub_row), _ptr(self.hub_chunk_ptr),
                                             _ptr(self.chunk_beg), _ptr(self.chunk_end), _ptr(ws), ws_bytes,
                                             _stream(dev)), "hub_fill")
            else:
                self.hub_row = self.hub_chunk_ptr = self.chunk_beg = self.chunk_end = None
        self.plan_bands(rank=self.col_rank() if self.n_hub else None)
        return self

    def col_rank(self) -> torch.Tensor:
        """int32 [max(col) + 1]: rank of every gathered row by the number of edges that gather it, most-gathered
        first, ties by ascending id (``gmlm_col_rank``)."""
        lib = _lib.load()
        dev = self.rowptr.device
        num_cols = int(self.col.max().item()) + 1 if self.nnz else 0
        with torch.cuda.device(dev):
            rank = torch.empty(num_cols, dtype=torch.int32, device=dev)
            ws_bytes = lib.gmlm_col_rank_workspace_bytes(num_cols)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            _lib.check(lib.gmlm_col_rank(_ptr(self.col), self.nnz, num_cols, _ptr(rank), _ptr(ws), ws_bytes,
                                         _stream(dev)), "col_rank")
        return rank

    @property
    def n_band_chunks(self) -> int:
        if self.band_plan is None:
            return 0
        return (int(self.band_plan.numel()) - self.n_hub - 2) // 2

    def plan_bands(self, band_shift: int = HUB_BAND_SHIFT, rank: Optional[torch.Tensor] = None):
        """The band-ordered hub plan next to the hub plan: every hub row's edges sorted by band key, cut into chunks
        at most ``hub_thresh`` long and at band boundaries, chunks ordered by band (``gmlm_hub_band_*``).  The key
        of a gathered row is ``rank[row]`` (``col_rank()``: band 0 holds the most-gathered rows, as ``plan_hubs``
        builds it), or the row id when ``rank`` is None."""
        self.hub_col = self.hub_w = self.band_plan = None
        if not self.n_hub:
            return self
        lib = _lib.load()
        dev = self.rowptr.device
        with torch.cuda.device(dev):
            hr = self.hub_row.long()
            lens = self.rowptr[hr + 1] - self.rowptr[hr]
            hub_off = torch.zeros(self.n_hub + 1, dtype=torch.int32, device=dev)
            torch.cumsum(lens, 0, out=hub_off[1:])
            n_edges = int(hub_off[-1].item())
            hub_col = torch.empty(n_edges, dtype=torch.int32, device=dev)
            hub_w = torch.empty(n_edges, dtype=torch.float32, device=dev) if self.w is not None and self.w.dim() == 1 else None
            chunk_ptr = torch.empty(self.n_hub + 1, dtype=torch.int32, device=dev)
            ws_bytes = lib.gmlm_hub_band_workspace_bytes(n_edges)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            n_band = C.c_int64(0)
            _lib.check(lib.gmlm_hub_band_sort(_ptr(self.rowptr), _ptr(self.col), _ptr(self.w if hub_w is not None else None),
                                              _ptr(rank), self.n_hub, _ptr(self.hub_row), _ptr(hub_off), n_edges,
                                              int(band_shift), self.hub_thresh, HUB_BAND_MIN_RUN, _ptr(hub_col),
                                              _ptr(hub_w), _ptr(chunk_ptr), C.byref(n_band), _ptr(ws), ws_bytes,
                                              _stream(dev)), "hub_band_sort")
            nb = int(n_band.value)
            band_plan = torch.empty(self.n_hub + 2 + 2 * nb, dtype=torch.int32, device=dev)
            band_plan[:self.n_hub + 1].copy_(chunk_ptr)
            _lib.check(lib.gmlm_hub_band_order(_ptr(hub_col), _ptr(rank), _ptr(hub_off), self.n_hub, n_edges, nb,
                                               int(band_shift), self.hub_thresh, HUB_BAND_MIN_RUN, _ptr(band_plan),
                                               _ptr(ws), ws_bytes, _stream(dev)), "hub_band_order")
        self.hub_col, self.hub_w, self.band_plan = hub_col, hub_w, band_plan
        return self


def build_csr(row: torch.Tensor, col: torch.Tensor, num_rows: int, num_cols: int, *,
              rel: Optional[torch.Tensor] = None, num_relations: int = 1,
              slot_of_rel: Optional[List[int]] = None, num_slots: int = 1,
              want_seg_of_edge: bool = False, hub_thresh: Optional[int] = None,
              quantum: Optional[int] = None, keep: Optional[torch.Tensor] = None):
    """CSR with segments ``row*num_slots + slot_of_rel[rel]`` and gather index ``col``.

    ``row``/``col``/``rel`` are int64 edge arrays (as in ``edge_index`` / ``edge_type``).
    Returns ``(CSR, seg_of_edge or None)``.  ``row`` is validated against ``num_rows`` and ``col``
    against ``num_cols`` (one host sync).  ``keep`` (bool [E], optional): edge-dropout mask fused into the
    build (N3) -- the result equals the CSR of ``edge_index[:, keep]``."""
    _require_cuda(row, "edge_index")
    if rel is not None and rel.dtype != torch.int64:
        rel = rel.long()
    rows_total = num_rows * num_slots
    slot_list = list(slot_of_rel) if slot_of_rel is not None else list(range(num_relations))
    from . import ops  # noqa: F401  (registers torch.ops.gmlm.*)
    rowptr, colv, perm, seg = torch.ops.gmlm.csr_build(row, col, rel, keep, int(num_rows), int(num_cols),
                                                       int(num_relations), [int(v) for v in slot_list], int(num_slots))
    if keep is not None:
        nnz = int(rowptr[-1].item())                 # kept edges; the dropped ones sorted behind them
        colv, perm = colv[:nnz], perm[:nnz]
    if not want_seg_of_edge:
        seg = None
    csr = CSR(rowptr=rowptr, col=colv, num_rows=rows_total, perm=perm)
    csr.plan_hubs(hub_thresh)
    csr.plan_groups(quantum)
    return csr, seg


def transpose_csr(row_of_edge: torch.Tensor, payload: torch.Tensor, num_rows: int, *,
                  fwd_rowptr: Optional[torch.Tensor] = None, edge_w: Optional[torch.Tensor] = None,
                  hub_thresh: Optional[int] = None, quantum: Optional[int] = None,
                  keep: Optional[torch.Tensor] = None) -> CSR:
    """CSR over ``row_of_edge`` (int64 [E]) whose gather index is ``payload`` (int32 [E], e.g. the
    forward segment of each edge); weights are 1/|fwd segment| or ``edge_w`` permuted.  ``keep``: as in
    ``build_csr``."""
    lib = _lib.load()
    dev = row_of_edge.device
    E = int(row_of_edge.numel())
    row_of_edge = row_of_edge.contiguous()
    with torch.cuda.device(dev):
        rowptr_t = torch.empty(num_rows + 1, dtype=torch.int32, device=dev)
        payload_t = torch.empty(E, dtype=torch.int32, device=dev)
        perm_t = torch.empty(E, dtype=torch.int32, device=dev)
        has_w = fwd_rowptr is not None or edge_w is not None
        w_t = torch.empty(E, dtype=torch.float32, device=dev) if has_w else None
        ws_bytes = lib.gmlm_csr_workspace_bytes(max(E, 1), num_rows)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        keep_u8 = None
        if keep is not None:
            keep_u8 = keep.contiguous().view(torch.uint8) if keep.dtype == torch.bool else (keep != 0).view(torch.uint8)
        _lib.check(lib.gmlm_csr_transpose(_ptr(row_of_edge), _ptr(payload), _ptr(edge_w), _ptr(fwd_rowptr),
                                          _ptr(keep_u8), E, num_rows, _ptr(rowptr_t), _ptr(payload_t), _ptr(w_t),
                                          _ptr(perm_t), _ptr(ws), ws_bytes, _stream(dev)), "csr_transpose")
    if keep is not None:
        nnz = int(rowptr_t[-1].item())
        payload_t, perm_t = payload_t[:nnz], perm_t[:nnz]
        w_t = w_t[:nnz] if w_t is not None else None
    csr = CSR(rowptr=rowptr_t, col=payload_t, num_rows=num_rows, w=w_t, perm=perm_t)
    csr.plan_hubs(hub_thresh)
    csr.plan_groups(quantum)
    return csr


@dataclass
class SegPlan:
    """Segment-compact view of a RelGraph (``RelGraph.seg_plan``): ``fwd`` rows = non-empty (dst, slot) segments in
    slot-major order (slot s owns rows ``slot_start[s] .. slot_start[s] + slot_count[s]``), gather index = source
    node; ``bwd`` rows = source nodes, gather index = compact row, weight = 1/|segment|; ``dst[k]`` = destination
    node of compact row k."""
    fwd: CSR
    bwd: CSR
    slot_start: List[int]
    slot_count: List[int]
    dst: torch.Tensor
    num_rows: int
    num_segments: int


@dataclass
class RelGraph:
    """Typed graph prepared for relational mean aggregation.

    ``fwd`` rows are the segments ``dst*num_slots + slot`` (slot = index of the relation among
    the populated ones), gather index = source node.  ``bwd`` rows are source nodes, gather
    index = forward segment, weight = 1/|segment|."""
    num_nodes: int                 # destination rows (== source rows for a whole graph)
    num_edges: int
    num_relations: int
    live_rels: List[int]
    fwd: CSR
    bwd: CSR
    num_src: int = -1              # source rows; > num_nodes for a partition with halo rows
    seg_of_edge: Optional[torch.Tensor] = None   # int32 [E] forward segment of each ORIGINAL edge (kept on request)
    _keepalive: list = field(default_factory=list, repr=False)
    _dst_plan: Optional[tuple] = field(default=None, repr=False)
    _seg_plan: Optional["SegPlan"] = field(default=None, repr=False)

    def __post_init__(self):
        if self.num_src < 0:
            self.num_src = self.num_nodes

    @property
    def num_slots(self) -> int:
        return len(self.live_rels)

    def dst_plan(self):
        """(fwd, bwd) CSR pair of the TRANSFORM-FIRST formulation (``gmlm_dst_plan``, include/gmlm_b200.h), built
        on first use and kept with the graph:

          fwd: rows = destination nodes; entries gather rows of Z = x @ [W_0|..|W_{S-1}|root] viewed as
               [num_src*(S+1), Fo] (col = src*(S+1)+slot, w = 1/|segment|; last entry = the node's own root slab)
          bwd: rows = (src, slot) pairs, i.e. the rows of dZ; entries gather rows of grad_out [N, Fo]."""
        if self._dst_plan is not None:
            return self._dst_plan
        lib = _lib.load()
        fwd = self.fwd
        dev = fwd.rowptr.device
        n, S, E = self.num_nodes, self.num_slots, self.num_edges
        with torch.cuda.device(dev):
            rowptr_d = torch.empty(n + 1, dtype=torch.int32, device=dev)
            col_d = torch.empty(E + n, dtype=torch.int32, device=dev)
            w_d = torch.empty(E + n, dtype=torch.float32, device=dev)
            dst_d = torch.empty(E + n, dtype=torch.int32, device=dev)
            _lib.check(lib.gmlm_dst_plan(_ptr(fwd.rowptr), _ptr(fwd.col), n, S, E, self.num_src, _ptr(rowptr_d),
                                         _ptr(col_d), _ptr(w_d), _ptr(dst_d), _stream(dev)), "dst_plan")
        f = CSR(rowptr=rowptr_d, col=col_d, num_rows=n, w=w_d, hub_thresh=fwd.hub_thresh)
        f.plan_hubs()
        f.plan_groups()
        b = transpose_csr(col_d.long(), dst_d, self.num_src * (S + 1), edge_w=w_d, hub_thresh=fwd.hub_thresh)
        self._dst_plan = (f, b)
        return self._dst_plan

    def seg_plan(self) -> "SegPlan":
        """The SEGMENT-COMPACT formulation (built on first use, kept with the graph): only the non-empty (dst, slot)
        segments become rows, ordered slot-major, so that the dense transform of relation s is ONE GEMM over the
        contiguous compact rows of slot s and multiplies no zero rows (79 % of the (dst, rel) rows of a power-law graph
        with degree-bucket relations are empty; 64 % on the Roman-empire shape).  The edges of a compact row keep their
        CSR order: its mean is bit-identical to the dense row's."""
        if self._seg_plan is not None:
            return self._seg_plan
        fwd, S, N = self.fwd, self.num_slots, self.num_nodes
        dev = fwd.rowptr.device
        rp = fwd.rowptr.long()
        lens = rp[1:] - rp[:-1]
        sid = torch.nonzero(lens > 0).flatten()                      # non-empty segments, dst-major
        slot, dst = sid % S, sid // S
        order = torch.argsort(slot * N + dst)                        # slot-major (keys are unique)
        cseg, dst_c, slot_c = sid[order], dst[order], slot[order]
        counts = torch.bincount(slot_c, minlength=S).cpu().tolist()  # one host read per graph
        # every slot starts on a multiple of 8 compact rows (a 16-byte boundary of the GEMM operand whatever the row
        # width); the padding rows are empty
        starts, rows = [], 0
        for c in counts:
            starts.append(rows)
            rows += (c + 7) // 8 * 8
        pos = torch.empty(cseg.numel(), dtype=torch.int64, device=dev)   # compact row of each non-empty segment
        off = 0
        for s_, c in enumerate(counts):
            pos[off:off + c] = torch.arange(starts[s_], starts[s_] + c, device=dev)
            off += c
        lens_c = torch.zeros(rows, dtype=torch.int64, device=dev)
        lens_c[pos] = lens[cseg]
        rowptr_c = torch.zeros(rows + 1, dtype=torch.int64, device=dev)
        rowptr_c[1:] = torch.cumsum(lens_c, 0)
        E = int(rowptr_c[-1].item()) if rows else 0
        old_start = torch.zeros(rows, dtype=torch.int64, device=dev)
        old_start[pos] = rp[cseg]
        e_idx = torch.repeat_interleave(old_start - rowptr_c[:-1], lens_c) + torch.arange(E, device=dev)
        col_c = fwd.col[e_idx].contiguous()
        crow = torch.repeat_interleave(torch.arange(rows, device=dev), lens_c).int()
        f = CSR(rowptr=rowptr_c.int(), col=col_c, num_rows=rows, hub_thresh=fwd.hub_thresh)
        f.plan_hubs()
        f.plan_groups()
        b = transpose_csr(col_c.long(), crow, self.num_src, fwd_rowptr=f.rowptr, hub_thresh=fwd.hub_thresh)
        dst_rows = torch.zeros(rows, dtype=torch.int64, device=dev)
        dst_rows[pos] = dst_c
        self._seg_plan = SegPlan(fwd=f, bwd=b, slot_start=starts, slot_count=counts, dst=dst_rows, num_rows=rows,
                                 num_segments=int(cseg.numel()))
        return self._seg_plan

    @property
    def num_nonempty_segments(self) -> int:
        if getattr(self, "_nseg", None) is None:
            rp = self.fwd.rowptr
            self._nseg = int((rp[1:] > rp[:-1]).sum().item())
        return self._nseg

    @staticmethod
    def build(edge_index: torch.Tensor, edge_type: Optional[torch.Tensor], num_nodes: int, num_relations: int,
              hub_thresh: Optional[int] = None, quantum: Optional[int] = None, num_src: Optional[int] = None,
              live_rels: Optional[List[int]] = None, keep_seg: bool = False,
              keep_mask: Optional[torch.Tensor] = None) -> "RelGraph":
        """``num_src`` > ``num_nodes`` builds the rectangular CSR of a destination-row partition
        (columns = local rows followed by halo rows).  ``live_rels`` pins the relation->slot
        layout (ranks of a partition must agree on it); default = the populated relations.
        ``keep_mask`` (bool [E]): the reference's edge dropout (``augment_graph``, main.py:832-837) fused into the
        build -- same graph as ``RelGraph.build(edge_index[:, keep_mask], edge_type[keep_mask], ...)`` without
        materialising the filtered edge list."""
        lib = _lib.load()
        n_src = num_nodes if num_src is None else int(num_src)
        _require_cuda(edge_index, "edge_index")
        if edge_index.dim() != 2 or edge_index.size(0) != 2:
            raise _lib.GmlmError(f"edge_index must have shape [2, E], got {tuple(edge_index.shape)}")
        edge_index = edge_index.long()
        src, dst = edge_index[0].contiguous(), edge_index[1].contiguous()
        E = int(src.numel())
        dev = edge_index.device
        if edge_type is None:
            live = [0]
            num_relations = max(1, num_relations)
        else:
            _require_cuda(edge_type, "edge_type")
            if edge_type.numel() != E:
                raise _lib.GmlmError(f"edge_type has {edge_type.numel()} entries for {E} edges")
            edge_type = edge_type.long().contiguous()
            with torch.cuda.device(dev):
                counts = torch.empty(num_relations, dtype=torch.int64, device=dev)
                keep_u8 = None
                if keep_mask is not None:
                    keep_u8 = (keep_mask.contiguous().view(torch.uint8) if keep_mask.dtype == torch.bool
                               else (keep_mask != 0).view(torch.uint8))
                _lib.check(lib.gmlm_relation_histogram(_ptr(edge_type), _ptr(keep_u8), E, num_relations, _ptr(counts),
                                                       _stream(dev)), "relation_histogram")
            counts_h = counts.cpu().tolist()
            live = [r for r, c in enumerate(counts_h) if c > 0]
            if live_rels is not None:
                if not set(live) <= set(live_rels):
                    raise _lib.GmlmError(f"live_rels {live_rels} does not cover the populated relations {live}")
                live = sorted(live_rels)
            n_kept = E if keep_mask is None else int(keep_mask.sum().item())
            if sum(counts_h) != n_kept:
                raise _lib.GmlmError(f"edge_type has values outside [0, {num_relations})")
            if not live:
                live = [0]
        slot_of_rel = [-1] * num_relations
        for s, r in enumerate(live):
            slot_of_rel[r] = s
        if edge_type is None:
            slot_of_rel[0] = 0
        fwd, seg = build_csr(dst, src, num_nodes, n_src, rel=edge_type, num_relations=num_relations,
                             slot_of_rel=slot_of_rel, num_slots=len(live), want_seg_of_edge=True,
                             hub_thresh=hub_thresh, quantum=quantum, keep=keep_mask)
        bwd = transpose_csr(src, seg, n_src, fwd_rowptr=fwd.rowptr, hub_thresh=hub_thresh, quantum=quantum,
                            keep=keep_mask)
        E = fwd.nnz                                    # kept edges
        return RelGraph(num_nodes=num_nodes, num_edges=E, num_relations=num_relations, live_rels=live, fwd=fwd,
                        bwd=bwd, num_src=n_src, seg_of_edge=seg if keep_seg else None)


# ------------------------------------------------------------------------------ cache
# The reference rebuilds its per-relation edge lists on every conv call.  Here the structure is built once
# per graph.  Two keys:
#   * identity  (data_ptr, _version, shape, ...) of the two tensors: the fast path, no device work;
#   * content   (shape, dtype, device, two 64-bit position-weighted checksums per tensor, `gmlm_checksum_i64`):
#     what makes the advertised one-line import swap hit -- the reference builds a FRESH edge_type tensor on
#     every get_graph_embeddings call (main.py:255), so identity alone would rebuild the CSR (two radix sorts,
#     four host syncs) per layer call.  A content lookup costs one pass over the indices and one host read.
# Alias entries hold strong references to their key tensors so that storage cannot be recycled under a stale
# identity key; `_version` catches in-place edits.  What they pin is bounded in BYTES as well as in count: under
# the import swap every call brings a fresh edge_type (8 bytes per edge -- 1.6 GB at 2e8 edges), so the oldest
# aliases are dropped once the table holds more than `GMLM_GRAPH_ALIAS_BYTES` (default 1 GiB; the newest alias
# always stays -- dropping an alias costs one checksum pass on the next call, never a rebuild).  Graphs are
# read-only after construction; the tables themselves are guarded by a lock (checkpoint recompute and backward
# run on autograd engine threads, one per device).
_CACHE: "OrderedDict[tuple, RelGraph]" = OrderedDict()           # content key -> graph
_ALIAS: "OrderedDict[tuple, tuple]" = OrderedDict()              # identity key -> (content key, keepalive tensors, bytes)
_CACHE_SIZE = int(os.environ.get("GMLM_GRAPH_CACHE", "4"))
_ALIAS_SIZE = 64
_ALIAS_BYTES = int(os.environ.get("GMLM_GRAPH_ALIAS_BYTES", str(1 << 30)))
_LOCK = threading.RLock()
cache_stats = {"identity_hits": 0, "content_hits": 0, "builds": 0}


def _alias_put(ikey: tuple, ckey: tuple, tensors: tuple) -> None:
    """Record identity key -> content key, keeping `tensors` alive; evict oldest-first by count and by bytes."""
    nbytes = sum(t.numel() * t.element_size() for t in tensors if t is not None)
    _ALIAS.pop(ikey, None)
    _ALIAS[ikey] = (ckey, tensors, nbytes)
    held = sum(v[2] for v in _ALIAS.values())
    while len(_ALIAS) > 1 and (len(_ALIAS) > _ALIAS_SIZE or held > _ALIAS_BYTES):
        held -= _ALIAS.popitem(last=False)[1][2]


def _tensor_key(t: Optional[torch.Tensor]):
    if t is None:
        return None
    return (t.data_ptr(), t._version, tuple(t.shape), tuple(t.stride()), t.dtype, str(t.device))


def _content_key(t: Optional[torch.Tensor]):
    if t is None:
        return None
    lib = _lib.load()
    x = t if (t.dtype == torch.int64 and t.is_contiguous()) else t.long().contiguous()
    with torch.cuda.device(x.device):
        out = torch.empty(2, dtype=torch.int64, device=x.device)
        _lib.check(lib.gmlm_checksum_i64(_ptr(x), x.numel(), _ptr(out), _stream(x.device)), "checksum")
    a, b = out.tolist()                                           # one host read
    return (tuple(t.shape), str(t.device), a, b)


def get_rel_graph(edge_index: torch.Tensor, edge_type: Optional[torch.Tensor], num_nodes: int,
                  num_relations: int) -> RelGraph:
    ikey = (_tensor_key(edge_index), _tensor_key(edge_type), int(num_nodes), int(num_relations))
    with _LOCK:
        hit = _ALIAS.get(ikey)
        if hit is not None and hit[0] in _CACHE:
            _ALIAS.move_to_end(ikey)
            _CACHE.move_to_end(hit[0])
            cache_stats["identity_hits"] += 1
            return _CACHE[hit[0]]
        _require_cuda(edge_index, "edge_index")
        ckey = (_content_key(edge_index), _content_key(edge_type), int(num_nodes), int(num_relations))
        g = _CACHE.get(ckey)
        if g is None:
            g = RelGraph.build(edge_index, edge_type, num_nodes, num_relations)
            _CACHE[ckey] = g
            cache_stats["builds"] += 1
            while len(_CACHE) > _CACHE_SIZE:
                _CACHE.popitem(last=False)
        else:
            _CACHE.move_to_end(ckey)
            cache_stats["content_hits"] += 1
        _alias_put(ikey, ckey, (edge_index, edge_type))           # keep the key tensors alive with the alias
        return g


def clear_graph_cache():
    with _LOCK:
        _CACHE.clear()
        _ALIAS.clear()
