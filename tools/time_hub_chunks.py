"""Time the hub path of the aggregation alone (chunk_kernel + hub_final_kernel, from torch.profiler kernel records)
and the whole call (every kernel of it) on the C5 / C4 graphs, forward (mean) and backward (weighted), for the
CSR-order chunk plan and the band-ordered plan keyed on the gathered row id ("id") or on its use rank ("rank",
CSR.col_rank) at several band shifts and hub thresholds.  Next to each time: the modelled gather traffic of the band
plan (distinct gathered rows per band pass x 512 bytes, against one row per hub edge), a model and not a DRAM
measurement.

    python tools/time_hub_chunks.py [--graphs c5 c4] [--keys id rank] [--iters 10] [--out profiles/x.jsonl]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import gmlm_b200 as G  # noqa: E402
from gmlm_b200 import _lib, synth  # noqa: E402
from gmlm_b200.graph import HUB_BAND_SHIFT  # noqa: E402

HUB_KERNELS = ("chunk_kernel", "hub_final_kernel")


def hub_ms(fn, iters):
    """Mean ms per call of the hub kernels of `fn` and of all its kernels ("call") (kernel records of
    torch.profiler)."""
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    tot = {k: 0.0 for k in HUB_KERNELS + ("call",)}
    for ev in prof.events():
        t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            tot["call"] += t
        for k in HUB_KERNELS:
            if k in ev.name and "tma" not in ev.name:
                tot[k] += t
    return {k: v / iters / 1e3 for k, v in tot.items()}


def gather_model(csr, shift, rank):
    """Hub edges and distinct gathered rows per band pass (chunks grouped by the band of their first edge)."""
    nh, nb = csr.n_hub, csr.n_band_chunks
    bp = csr.band_plan.long()
    cut = bp[nh + 1:nh + 2 + nb]
    lens = cut[1:] - cut[:-1]
    band_key = csr.hub_col.long() if rank is None else rank.long()[csr.hub_col.long()]
    first_band = band_key[cut[:-1]] >> shift
    band_of_edge = torch.repeat_interleave(first_band, lens)
    key = band_of_edge * (int(csr.hub_col.max().item()) + 1) + csr.hub_col.long()
    distinct = int(torch.unique(key).numel())
    return {"hub_edges": int(csr.hub_col.numel()), "distinct_rows_per_band_pass": distinct,
            "modelled_gather_gb_banded": distinct * 512 / 1e9, "modelled_gather_gb_one_row_per_edge":
            int(csr.hub_col.numel()) * 512 / 1e9, "chunks": nb, "chunks_csr_order": csr.n_chunks}


def without_bands(csr):
    c = G.graph.CSR(**{k: getattr(csr, k) for k in csr.__dataclass_fields__})
    c.hub_col = c.hub_w = c.band_plan = None
    return c


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graphs", nargs="+", default=["c5", "c4"])
    ap.add_argument("--shifts", nargs="+", type=int, default=[16, 17, 18])
    ap.add_argument("--keys", nargs="+", default=["id", "rank"], choices=["id", "rank"])
    ap.add_argument("--threshs", nargs="+", type=int, default=[256, 128, 64])
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    lines = []

    def emit(d):
        d["gpu"] = gpu
        print(json.dumps(d), flush=True)
        lines.append(d)

    for key in args.graphs:
        w = synth.WORKLOADS[key]
        ei = synth.make_graph(w, device=dev)
        et = G.edge_type_from_degree(ei, w.num_nodes)
        g = G.get_rel_graph(ei, et, w.num_nodes, 5)
        x = synth.make_features(w.num_nodes, 256, device=dev, dtype=torch.bfloat16)
        gh = synth.make_features(w.num_nodes * g.num_slots, 256, device=dev, seed=7, dtype=torch.bfloat16)
        h_buf = torch.empty((w.num_nodes * g.num_slots, 256), dtype=torch.bfloat16, device=dev)
        gx_buf = torch.empty((w.num_nodes, 256), dtype=torch.bfloat16, device=dev)
        for thresh in args.threshs:
            for csr in (g.fwd, g.bwd):
                if csr.hub_thresh != thresh:
                    csr.plan_hubs(thresh)
            for name, csr, inp, buf, mode in (("fwd", g.fwd, x, h_buf, _lib.AGG_MEAN),
                                               ("bwd", g.bwd, gh, gx_buf, _lib.AGG_WEIGHTED)):
                plain = without_bands(csr)
                emit({"graph": key, "dir": name, "hub_thresh": thresh, "plan": "csr_order",
                      "ms": hub_ms(lambda: G.spmm(inp, plain, mode, out=buf), args.iters),
                      "hub_rows": csr.n_hub, "chunks": csr.n_chunks})
                for band_key in args.keys:
                    for shift in (args.shifts if thresh == args.threshs[0] else [HUB_BAND_SHIFT]):
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        rank = csr.col_rank() if band_key == "rank" else None
                        torch.cuda.synchronize()
                        t_rank = time.perf_counter() - t0
                        csr.plan_bands(shift, rank=rank)
                        torch.cuda.synchronize()
                        t_plan = time.perf_counter() - t0
                        d = {"graph": key, "dir": name, "hub_thresh": thresh, "plan": "banded", "band_key": band_key,
                             "band_shift": shift, "ms": hub_ms(lambda: G.spmm(inp, csr, mode, out=buf), args.iters),
                             "plan_build_s": t_plan, "rank_build_s": t_rank,
                             "plan_bytes": 4 * (csr.hub_col.numel() + csr.band_plan.numel()) +
                             (4 * csr.hub_w.numel() if csr.hub_w is not None else 0),
                             "rank_bytes": 4 * rank.numel() if rank is not None else 0}
                        d.update(model=gather_model(csr, shift, rank))
                        emit(d)
                        del rank
                csr.plan_hubs(csr.hub_thresh)
            for csr in (g.fwd, g.bwd):
                csr.plan_hubs(G.graph.DEFAULT_HUB_THRESH)
        del g, ei, et, x, gh, h_buf, gx_buf
        G.clear_graph_cache()
        torch.cuda.empty_cache()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(d) + "\n" for d in lines))


if __name__ == "__main__":
    main()
