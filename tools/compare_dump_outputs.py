"""Compare the outputs two builds wrote with ``bench.py --dump-outputs DIR`` (h and grad_x of the last timed step,
the same sampled rows in both), split by whether a sampled row is a hub row of its CSR (hub rows sum their chunks
in plan order, every other row in CSR order).  Rebuilds the workload's graph to know the hub rows, so it needs the
GPU.  One JSON line per output.

    python tools/compare_dump_outputs.py DIR_A DIR_B [--workload c5] [--out profiles/x.jsonl]
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import gmlm_b200 as G  # noqa: E402
from bench import DUMP_BYTES  # noqa: E402
from gmlm_b200 import synth  # noqa: E402


def sampled_rows(rows, width, n_outputs):
    """The row ids bench.dump_outputs keeps (same generator and seed)."""
    k = min(rows, max(1, (DUMP_BYTES // n_outputs) // (4 * width)))
    if k == rows:
        return torch.arange(rows)
    stride = rows // k
    return torch.arange(k) * stride + torch.randint(0, stride, (k,), generator=torch.Generator().manual_seed(0))


def bf16_order(a):
    """bf16 values (held in float32) -> integers whose differences count bf16 ulps."""
    u = a.view(np.uint32) >> 16
    mag = (u & 0x7FFF).astype(np.int64)
    return np.where(u & 0x8000, -mag, mag)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("dir_a")
    ap.add_argument("dir_b")
    ap.add_argument("--workload", default="c5")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    w = synth.WORKLOADS[args.workload]
    dev = torch.device("cuda:0")
    ei = synth.make_graph(w, device=dev)
    g = G.get_rel_graph(ei, G.edge_type_from_degree(ei, w.num_nodes), w.num_nodes, 5)
    lines = []
    for name, csr in (("h", g.fwd), ("grad_x", g.bwd)):
        a = np.load(Path(args.dir_a) / f"{name}.npy")
        b = np.load(Path(args.dir_b) / f"{name}.npy")
        idx = sampled_rows(csr.num_rows, a.shape[1], 2)
        assert a.shape == b.shape and a.shape[0] == idx.numel()
        hub = torch.zeros(csr.num_rows, dtype=torch.bool)
        if csr.n_hub:
            hub[csr.hub_row.long().cpu()] = True
        hub = hub[idx].numpy()
        diff = np.abs(a - b)
        ulp = np.abs(bf16_order(a) - bf16_order(b))
        rel = diff[hub] / np.maximum(np.abs(a[hub]), 1e-30)
        d = {"output": name, "rows_sampled": int(idx.numel()), "hub_rows_sampled": int(hub.sum()),
             "nonhub_rows_identical": bool(np.array_equal(a[~hub], b[~hub])),
             "hub_elements_differing_frac": float((diff[hub] > 0).mean()) if hub.any() else 0.0,
             "all_elements_differing_frac": float((diff > 0).mean()),
             "max_ulp_bf16_hub": int(ulp[hub].max()) if hub.any() else 0,
             "max_abs_diff": float(diff.max()), "max_rel_diff_hub": float(rel.max()) if hub.any() else 0.0}
        print(json.dumps(d), flush=True)
        lines.append(d)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(d) + "\n" for d in lines))


if __name__ == "__main__":
    main()
