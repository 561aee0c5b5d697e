#!/usr/bin/env python
"""bench.py — message-passing edges/s (fwd+bwd) of the GMLM GNN-encoder hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c4|c5|c2|c3]
                    [--dump-outputs DIR]

One "step" = one forward + one backward propagate of the F=256 RGCN mean aggregation (the
kernel pair SURVEY §8(d) defines the algorithmic bytes for: 1162 B/edge in bf16) over the whole
synthetic graph.  Every N runs BASELINE.json configs[4]'s graph (10M nodes / 200M edges, bf16): whole
on one GPU at N=1 (the denominator of the 1/2/4/8 scaling the metric names; the same line carries
configs[3] — 2M / 40M, the HBM-roofline study — under "c4"), destination-row partitioned with the
NVLink halo exchange of gmlm_b200/partition.py at N>1.  Rank 0 prints ONE JSON line.

`--impl reference` times the reference's CPU implementation of the same path — the oracle
port of the torch_geometric index_select/scatter path (oracle/pyg_ref.py; PyG itself is not
installable here) — on the host cores, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

FALLBACK_HBM_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback
NVLINK_GBS = 770.0          # measured peer copy per direction per GPU (same guide)


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(n_nodes, n_edges, feat, esize, live_rels):
    """SURVEY §8(d): bytes one propagate must move (int32 CSR, no credit for cache hits)."""
    fwd = n_edges * feat * esize + 4 * n_edges + 4 * (n_nodes * live_rels + 1) + n_nodes * live_rels * feat * esize
    bwd = n_edges * feat * esize + 4 * n_edges + n_edges + 4 * (n_nodes + 1) + n_nodes * feat * esize
    return fwd, bwd


_ONES_CACHE = {}


def _ones_like(y):
    """Upstream gradient of the context legs, created once per shape: in training it comes out of the loss; a fresh
    `ones_like` per step would put a [N, out] fill (0.8 ms at 2M x 768) inside every timed step."""
    key = (tuple(y.shape), y.dtype, y.device)
    t = _ONES_CACHE.get(key)
    if t is None:
        if len(_ONES_CACHE) > 4:
            _ONES_CACHE.clear()
        t = _ONES_CACHE[key] = torch.ones_like(y)
    return t


DUMP_BYTES = 32 << 20


def dump_outputs(out_dir, outputs):
    """Write each output of the timed path as <out_dir>/<name>.npy in float32.  An output larger than its share of
    DUMP_BYTES keeps a fixed sample of rows (one row drawn by a seeded CPU generator from each of k equal strides):
    the same rows for every run with the same arguments, so two builds can be compared output for output."""
    import numpy as np
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    share = DUMP_BYTES // len(outputs)
    for name, t in outputs.items():
        rows, width = t.shape[0], t[0].numel() if t.shape[0] else 1
        k = min(rows, max(1, share // (4 * width)))
        if k < rows:
            stride = rows // k
            idx = torch.arange(k) * stride + torch.randint(0, stride, (k,), generator=torch.Generator().manual_seed(0))
            t = t[idx.to(t.device)]
        np.save(out_dir / f"{name}.npy", t.float().cpu().numpy())
        print(f"dumped {name}: {k} of {rows} rows, float32", file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [s.strip() for s in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- CPU reference arm
def cpu_reference_step_factory(sample_nodes: int, sample_edges: int, feat: int):
    """The oracle port of the reference path on host cores: per-relation index_select +
    index_add_ mean (fwd) and its autograd backward, fp32 (what torch_geometric runs on CPU)."""
    from gmlm_b200 import synth
    from oracle import edge_type_bucket_ref, rgcn_propagate_mean_ref

    ei = synth.rmat_edges(sample_nodes, sample_edges, device="cpu", seed=42)
    et = edge_type_bucket_ref(ei, sample_nodes)
    x = synth.make_features(sample_nodes, feat, device="cpu", seed=42)
    rels = sorted(set(et.unique().tolist()))
    per_rel = [(ei[0, et == r].contiguous(), ei[1, et == r].contiguous()) for r in rels]
    gh = [torch.randn(sample_nodes, feat) for _ in rels]

    def step():
        xg = x.detach().requires_grad_(True)
        outs = [rgcn_propagate_mean_ref(xg, s, d, sample_nodes) for s, d in per_rel]
        torch.autograd.backward(outs, gh)
        return xg.grad

    return step


def time_cpu_reference(steps: int, warmup: int, sample_nodes: int, sample_edges: int, feat: int):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step = cpu_reference_step_factory(sample_nodes, sample_edges, feat)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return sample_edges / dt, dt * 1e3, cores


def baseline_extras(ei, x, et, n, e, gpu_typing_s, dev):
    """Two more reported baselines of SURVEY §8(d), same leg as cpu_baseline (the only place bench.py runs
    oracle code): (i) the edge-typing step — the reference's verbatim per-edge Python loop
    (main.py:253-267) on a bounded sample and its vectorised form on the host, next to our kernel;
    (ii) the stock-PyTorch path (index_select + index_add_ atomics per relation, what torch_geometric
    executes) run ON THE B200 on the full workload — what the reference would get from the same GPU."""
    from oracle import edge_type_bucket_ref, edge_type_loop_ref, rgcn_propagate_mean_ref
    out = {}
    try:
        m = min(e, 20_000)
        ei_s = ei[:, :m].cpu()
        t0 = time.perf_counter()
        edge_type_loop_ref(ei_s, n)
        loop_s = time.perf_counter() - t0
        ei_c = ei.cpu() if e <= 50_000_000 else ei[:, :50_000_000].cpu()
        t0 = time.perf_counter()
        edge_type_bucket_ref(ei_c, n)
        vec_s = time.perf_counter() - t0
        out["edge_typing"] = {"reference_python_loop_us_per_edge": loop_s / max(m, 1) * 1e6,
                              "reference_loop_extrapolated_s": loop_s / max(m, 1) * e,
                              "vectorised_cpu_s": vec_s * (e / max(ei_c.size(1), 1)),
                              "our_kernel_s": gpu_typing_s, "sample_edges_for_loop": m}
    except Exception as ex:
        out["edge_typing"] = {"error": repr(ex)[:200]}
    try:
        rels = sorted(torch.unique(et).tolist())
        per_rel = [(ei[0, et == r].contiguous(), ei[1, et == r].contiguous()) for r in rels]
        gh = [torch.randn(n, x.size(1), device=dev, dtype=x.dtype) for _ in rels]

        def step():
            xg = x.detach().requires_grad_(True)
            outs = [rgcn_propagate_mean_ref(xg, s_, d_, n) for s_, d_ in per_rel]
            torch.autograd.backward(outs, gh)

        step()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(3):
            step()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / 3
        out["stock_torch_on_gpu"] = {"value": e / (ms * 1e-3), "unit": "edges/s", "ms_per_step": ms,
                                     "what": "oracle port (index_select + index_add_ per relation, autograd "
                                             "backward) on the same B200, same graph and dtype"}
        del per_rel, gh
        torch.cuda.empty_cache()
    except Exception as ex:
        out["stock_torch_on_gpu"] = {"error": repr(ex)[:200]}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from gmlm_b200 import synth
    w = synth.WORKLOADS[args.workload]
    sn, se = args.cpu_sample_nodes, args.cpu_sample_edges
    eps, ms, cores = time_cpu_reference(args.steps, args.warmup, sn, se, w.feat)
    sample = (f"R-MAT sample {sn} nodes / {se} edges / F={w.feat} fp32 of workload {w.key}, fwd+bwd of the "
              f"per-relation index_select+index_add_ mean (oracle port of torch_geometric RGCNConv.propagate)")
    line = {
        "impl": "reference", "metric": "message-passing edges/sec fwd+bwd", "value": eps, "unit": "edges/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong" if w.key == "c5" else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": w.title, "feat": w.feat, "sample": sample},
        "cpu_baseline": {"value": eps, "unit": "edges/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": eps, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- our arm, one GPU
def measure_single(args, key: str, extras: bool, with_cpu: bool, dump_dir=None):
    """One workload on one GPU -> the fields of the JSON line (value, roofline, e2e, context legs).  With
    ``dump_dir``, the last timed step's outputs are written there (dump_outputs)."""
    import gmlm_b200 as G
    from gmlm_b200 import _lib, synth

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback); use --impl reference"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    w = synth.WORKLOADS[key]
    n = int(w.num_nodes * args.scale)
    e = int(w.num_edges * args.scale)
    feat = w.feat
    dtype = torch.bfloat16 if w.dtype == "bf16" else torch.float32
    esize = 2 if dtype == torch.bfloat16 else 4

    t0 = time.perf_counter()
    ei = synth.make_graph(w, device=dev, num_nodes=n, num_edges=e)
    x = synth.make_features(n, feat, device=dev, dtype=dtype)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t0

    t0 = time.perf_counter()
    et = G.edge_type_from_degree(ei, n)
    torch.cuda.synchronize()
    t_type = time.perf_counter() - t0
    t0 = time.perf_counter()
    g = G.get_rel_graph(ei, et, n, 5)
    torch.cuda.synchronize()
    t_csr = time.perf_counter() - t0
    S = g.num_slots
    gh = synth.make_features(n * S, feat, device=dev, seed=7, dtype=dtype)     # upstream grad of H

    launches_per_step = 2 + (2 if g.fwd.n_hub else 0) + (2 if g.bwd.n_hub else 0)

    # the two outputs live in buffers allocated ONCE (as a training loop's steady state does through the caching
    # allocator): a fresh 20 GB `torch.empty` per call made single steps of the timed loop stall for ~100 ms whenever
    # the allocator had to return cached blocks to the driver (cudaFree synchronises) -- one run in four measured a
    # 28-30 ms forward mean against 17.7 ms for exactly the same kernels (per-step min / max are in the line)
    h_buf = torch.empty((n * S, feat), dtype=dtype, device=dev)
    gx_buf = torch.empty((n, feat), dtype=dtype, device=dev)

    def step():
        h = G.spmm(x, g.fwd, _lib.AGG_MEAN, out=h_buf)             # A5  forward propagate (all relations)
        gx = G.spmm(gh, g.bwd, _lib.AGG_WEIGHTED, out=gx_buf)      # A14 backward propagate
        return h, gx

    sampler = ClockSampler(0)
    sampler.start()               # before the warm-up: nvidia-smi's NVML start-up must not land in the timed region
    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    time.sleep(0.3)
    for _ in range(2):
        step()
    torch.cuda.synchronize()

    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    t_start = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    torch.cuda.nvtx.range_push("timed")      # ncu --nvtx --nvtx-include "timed/" lists exactly these launches
    t_start.record()
    for k in range(args.steps):
        ev[k][0].record()
        h = G.spmm(x, g.fwd, _lib.AGG_MEAN, out=h_buf)
        ev[k][1].record()
        gx = G.spmm(gh, g.bwd, _lib.AGG_WEIGHTED, out=gx_buf)
        ev[k][2].record()
    t_end.record()
    torch.cuda.synchronize()
    torch.cuda.nvtx.range_pop()
    clocks = sampler.stop()
    if dump_dir is not None:
        dump_outputs(dump_dir, {"h": h, "grad_x": gx})
    total_ms = t_start.elapsed_time(t_end)
    ms_per_step = total_ms / args.steps
    fwd_all = [a.elapsed_time(b) for a, b, _ in ev]
    bwd_all = [b.elapsed_time(c) for _, b, c in ev]
    fwd_ms = statistics.mean(fwd_all)
    bwd_ms = statistics.mean(bwd_all)
    value = e / (ms_per_step * 1e-3)

    fwd_b, bwd_b = algorithmic_bytes(n, e, feat, esize, S)
    peak, peak_src = peaks()
    traffic = traffic_bwd = None
    tj = ROOT / "profiles" / "traffic.json"
    if tj.exists() and args.scale == 1.0:
        try:
            tr = json.loads(tj.read_text())
            traffic, traffic_bwd = tr.get(f"{w.key}_fwd"), tr.get(f"{w.key}_bwd")
        except Exception:
            traffic = traffic_bwd = None
    roof = {"bound": "hbm", "kernel": "forward aggregate (A5): rows_kernel + chunk_kernel + hub_final_kernel",
            "achieved": fwd_b / (fwd_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
            "frac": fwd_b / (fwd_ms * 1e-3) / 1e9 / peak, "traffic": traffic, "peak_source": peak_src,
            "algorithmic_bytes": fwd_b, "ms": fwd_ms, "ms_min_max": [min(fwd_all), max(fwd_all)]}
    if traffic:
        roof["traffic_source"] = ("stored ncu figure (dram__bytes_read.sum + dram__bytes_write.sum of the same kernels on "
                                  "this workload, profiles/traffic.json), NOT measured in this run")
        roof["dram_gbs"] = traffic / (fwd_ms * 1e-3) / 1e9
        roof["note"] = ("achieved counts ALGORITHMIC bytes (SURVEY §8d: no credit for cache hits); on this power-law "
                        "graph the 126 MB L2 serves the hub source rows, so DRAM traffic (ncu, `traffic`) is well below "
                        "the algorithmic bytes and frac can exceed 1. On a uniform-random graph of the same size "
                        "(L2 hit rate ~12 %) the same kernels measure 1.02x the copy peak (profiles/).")
    roof_bwd = {"bound": "hbm", "kernel": "backward aggregate (A14): rows_kernel<weighted> + chunk_kernel<weighted> + hub_final_kernel",
                "achieved": bwd_b / (bwd_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": bwd_b / (bwd_ms * 1e-3) / 1e9 / peak, "traffic": traffic_bwd, "algorithmic_bytes": bwd_b,
                "ms": bwd_ms}
    if traffic_bwd:
        roof_bwd["dram_gbs"] = traffic_bwd / (bwd_ms * 1e-3) / 1e9
    roof_step = {"achieved": (fwd_b + bwd_b) / (ms_per_step * 1e-3) / 1e9, "peak": peak,
                 "frac": (fwd_b + bwd_b) / (ms_per_step * 1e-3) / 1e9 / peak, "unit": "GB/s"}

    del h, gx, h_buf, gx_buf                     # 25 GB on C5: the legs below allocate their own
    # ---- e2e: public autograd API, x from pinned host memory every step, scalar result read back
    #      (a copy stream double-buffers the next step's H2D under the current step's kernels)
    x_host = x.cpu().pin_memory()
    bufs = [torch.empty_like(x), torch.empty_like(x)]
    e2e_steps = max(3, min(args.steps, 10))
    res_host = torch.empty(e2e_steps + 2, dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream()
    main = torch.cuda.current_stream()
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    freed = [torch.cuda.Event(), torch.cuda.Event()]

    def issue_copy(k):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[k % 2])
            bufs[k % 2].copy_(x_host, non_blocking=True)
            ready[k % 2].record(copy_stream)

    def e2e_run(steps):
        for ev_ in freed:
            ev_.record(main)
        issue_copy(0)
        for k in range(steps):
            if k + 1 < steps:
                issue_copy(k + 1)
            main.wait_event(ready[k % 2])
            xg = bufs[k % 2].detach().requires_grad_(True)
            out = G.rgcn_aggregate(xg, g)                      # public autograd API
            out.backward(gh.view_as(out))
            res_host[k:k + 1].copy_(xg.grad[:: max(1, n // 4096)].float().sum().reshape(1), non_blocking=True)
            freed[k % 2].record(main)

    e2e_run(2)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    e2e_run(e2e_steps)
    b.record()
    torch.cuda.synchronize()
    e2e_ms = a.elapsed_time(b) / e2e_steps
    e2e = {"value": e / (e2e_ms * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": x_host.numel() * esize,
           "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms,
           "note": "x copied from pinned host memory every step (double-buffered on a copy stream), fwd+bwd through "
                   "rgcn_aggregate autograd, scalar result read back; graph/CSR resident (static graph, as in the "
                   "reference). PCIe-bound: %.2f GB per step" % (x_host.numel() * esize / 1e9)}
    del bufs, x_host

    # ---- full message-passing layer (A5+A6+A7 fwd+bwd) for context
    layer = None
    if extras and not args.no_layer:
        try:
            conv = G.RGCNConv(feat, w.hidden, 5, 30, out_dtype=dtype).to(dev)
            norm = G.GraphNorm(w.hidden).to(dev)
            xg = x.detach().requires_grad_(True)

            def layer_step():
                y = norm(conv(xg, g), fuse_gelu=True)
                y.backward(_ones_like(y))
                xg.grad = None
                conv.zero_grad(set_to_none=True)     # as optimizer.zero_grad() does every step (main.py:439,530):
                norm.zero_grad(set_to_none=True)     # gradients are written, not accumulated into last step's

            for _ in range(3):
                layer_step()
            torch.cuda.synchronize()
            a.record()
            for _ in range(5):
                layer_step()
            b.record()
            torch.cuda.synchronize()
            lms = a.elapsed_time(b) / 5
            layer = {"ms_fwd_bwd": lms, "edges_per_s": e / (lms * 1e-3),
                     "what": f"RGCNConv({feat}->{w.hidden}) + GraphNorm + GELU fwd+bwd incl. weight grads"}
        except Exception as ex:  # context only; never hides the headline
            layer = {"error": repr(ex)[:200]}

    # ---- whole GNN encoder (get_graph_embeddings, main.py:250-320): four layers + residuals + fusion,
    #      forward + backward ("epoch" of the encoder on this graph); edges/s counts 4*E per pass
    encoder = None
    if extras and not args.no_layer:
        try:
            del gh
            torch.cuda.empty_cache()
            enc = G.GraphEncoder(feat, w.hidden, 768, dropout_rate=0.0, act_dtype=dtype).to(dev)
            if dtype == torch.bfloat16:
                enc.residual_proj1.to(dtype), enc.residual_proj2.to(dtype), enc.multi_scale_fusion.to(dtype)
            xg = x.detach().requires_grad_(True)

            # fp32 workloads (the reference's own dataset shapes) run the encoder under autocast, as the
            # reference's training loops do (main.py:446,543); the bf16 study runs bf16 end to end
            use_autocast = dtype == torch.float32

            def enc_step():
                with torch.amp.autocast("cuda", enabled=use_autocast):
                    y = enc.get_graph_embeddings(xg, ei, et)
                y.backward(_ones_like(y))
                xg.grad = None
                enc.zero_grad(set_to_none=True)      # optimizer.zero_grad() of the reference's loops (main.py:439,530)

            for _ in range(2):
                enc_step()
            torch.cuda.synchronize()
            a.record()
            for _ in range(3):
                enc_step()
            b.record()
            torch.cuda.synchronize()
            ems = a.elapsed_time(b) / 3
            encoder = {"ms_fwd_bwd": ems, "edges_per_s": 4 * e / (ems * 1e-3), "hidden_channels": w.hidden,
                       "autocast": use_autocast,
                       "what": "GraphEncoder.get_graph_embeddings fwd+bwd: 4x(RGCNConv+GraphNorm+GELU), residual "
                               "projections, MultiScaleFusion(->768); edges/s counts the 4 propagates"}
            del enc
        except Exception as ex:
            encoder = {"error": repr(ex)[:300]}

    cpu = None
    if with_cpu and not args.no_cpu_baseline:
        eps, cms, cores = time_cpu_reference(2, 1, args.cpu_sample_nodes, args.cpu_sample_edges, feat)
        cpu = {"value": eps, "unit": "edges/s", "cores": cores, "kind": "port",
               "sample": f"R-MAT {args.cpu_sample_nodes} nodes / {args.cpu_sample_edges} edges, F={feat} fp32, "
                         f"fwd+bwd, oracle port of torch_geometric propagate (index_select+index_add_), "
                         f"{cms:.0f} ms/step, best-effort 2 steps after 1 warm-up"}
        cpu.update(baseline_extras(ei, x, et, n, e, t_type, dev))

    line = {
        "metric": "message-passing edges/sec fwd+bwd", "value": value, "unit": "edges/s", "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong" if key == "c5" else "weak", "vs_baseline": None, "dtype": w.dtype, "data": "synthetic",
        "config": {"workload": w.title, "num_nodes": n, "num_edges": e, "feat": feat, "live_relations": S,
                   "generator": f"R-MAT{synth.RMAT_ABCD} seed 42, ids mod N" if w.generator == "rmat" else "uniform seed 42",
                   "l2": "inputs exceed L2 (x %.2f GB, H %.2f GB per step; no flush needed)" % (
                       n * feat * esize / 1e9, n * S * feat * esize / 1e9),
                   "step": "fwd aggregate (A5) + bwd aggregate (A14), F=%d" % feat,
                   "hub_thresh": g.fwd.hub_thresh, "hub_rows_fwd": g.fwd.n_hub, "hub_rows_bwd": g.bwd.n_hub},
        "roofline": roof, "roofline_bwd": roof_bwd, "roofline_step": roof_step,
        "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches_per_step * args.steps,
        "clocks": clocks, "layer": layer, "encoder": encoder,
        "setup_s": {"generate": t_gen, "edge_typing": t_type, "csr_build": t_csr},
    }
    del g, ei, et, x
    G.clear_graph_cache()
    torch.cuda.empty_cache()
    return line


# ----------------------------------------------------------------------------- the reference's own dataset shapes
def measure_small(args, key: str, with_stock: bool):
    """BASELINE.json configs[1] / configs[2]: the GNN encoder of main.py:250-320 with the shipped widths
    (hidden_channels = 512) on a Roman-empire- / Amazon-ratings-shaped graph, forward + backward under
    torch.amp.autocast exactly as the reference's training loops call it (main.py:446,543); configs[2] adds a
    GATConv(300 -> 8 x 64) layer (the edge-softmax variant north_star names).  These graphs fit in L2, so the
    figure is TIME (an encoder pass; a contrastive pre-training epoch runs two, main.py:447-448), not HBM
    fraction.  `stock_torch_on_gpu` = the oracle modules (index_select / index_add_ / scatter ops, what
    torch_geometric executes) on the same B200, same inputs -- part of the baseline leg."""
    import gmlm_b200 as G
    from gmlm_b200 import synth

    dev = torch.device("cuda:0")
    w = synth.WORKLOADS[key]
    n, e, feat = w.num_nodes, w.num_edges, w.feat
    ei = synth.make_graph(w, device=dev)
    x = synth.make_features(n, feat, device=dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timeit(fn, warm=3, iters=10):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters

    out = {"workload": w.title, "num_nodes": n, "num_edges": e, "feat": feat, "hidden_channels": w.hidden}
    torch.manual_seed(0)
    enc = G.GraphEncoder(feat, w.hidden, 768, dropout_rate=0.0).to(dev)
    xg = x.detach().requires_grad_(True)

    def enc_step(m=enc):
        with torch.amp.autocast("cuda"):
            y = m.get_graph_embeddings(xg, ei)
        y.backward(_ones_like(y))
        xg.grad = None
        m.zero_grad(set_to_none=True)                # optimizer.zero_grad() of the reference's loops (main.py:439,530)

    ms = timeit(enc_step)
    out["encoder_ms_fwd_bwd_eager"] = ms
    # the same step captured once as a CUDA graph and replayed (gmlm_b200.GraphedEncoderStep): what a training loop on
    # these static small graphs runs; the input copy into the captured buffer is inside the timed call
    try:
        enc.zero_grad(set_to_none=True)
        step = G.GraphedEncoderStep(enc, x, ei, autocast=True, x_requires_grad=True)
        gms = timeit(lambda: step(x))
        out["encoder_ms_fwd_bwd"] = gms
        out["encoder_mode"] = "cuda_graph (one launch per step); eager figure beside it"
        del step
        enc.zero_grad(set_to_none=True)
        ms = min(ms, gms)
    except Exception as ex:  # context leg: fall back to the eager figure, say why
        out["encoder_ms_fwd_bwd"] = ms
        out["encoder_mode"] = "eager (cuda graph capture failed: %s)" % repr(ex)[:160]
    ms = out["encoder_ms_fwd_bwd"]
    out["pretrain_epoch_encoder_ms"] = 2 * ms
    out["encoder_edges_per_s"] = 4 * e / (ms * 1e-3)
    gat = None
    if key == "c3":
        gat = G.GATConv(feat, 64, heads=8).to(dev)

        def gat_step(m=gat):
            y = m(xg, ei)
            y.backward(_ones_like(y))
            xg.grad = None
            m.zero_grad(set_to_none=True)

        out["gat_layer_ms_fwd_bwd"] = timeit(gat_step)
        out["gat_layer_what"] = "GATConv(300 -> 8 heads x 64): fused one-pass edge-softmax aggregation, fp32"
    if with_stock:
        try:
            from oracle import EncoderRef, GATConvRef
            torch.manual_seed(0)
            ref = EncoderRef(feat, w.hidden, 768, dropout_rate=0.0, use_checkpoint=False).to(dev)

            def ref_step():
                with torch.amp.autocast("cuda"):
                    y = ref(xg, ei)
                y.backward(_ones_like(y))
                xg.grad = None
                ref.zero_grad(set_to_none=True)

            stock = {"encoder_ms_fwd_bwd": timeit(ref_step, warm=2, iters=5),
                     "what": "oracle EncoderRef (vectorised edge typing + per-relation index_select/index_add_ "
                             "RGCN, stock GraphNorm ops) on the same B200 under autocast; the reference's own "
                             "per-edge Python typing loop is NOT included (it alone costs seconds per call)"}
            if gat is not None:
                gref = GATConvRef(feat, 64, heads=8).to(dev)

                def gref_step():
                    y = gref(xg, ei)
                    y.backward(_ones_like(y))
                    xg.grad = None
                    gref.zero_grad(set_to_none=True)

                stock["gat_layer_ms_fwd_bwd"] = timeit(gref_step, warm=2, iters=5)
            out["stock_torch_on_gpu"] = stock
            del ref
        except Exception as ex:
            out["stock_torch_on_gpu"] = {"error": repr(ex)[:200]}
    del enc
    G.clear_graph_cache()
    torch.cuda.empty_cache()
    return out


def run_single(args):
    """N=1.  Default: BASELINE.json configs[4]'s graph (10M nodes / 200M edges) whole on one GPU — the
    denominator of the 1/2/4/8-GPU scaling the metric names — followed by configs[3] (2M / 40M, the
    HBM-roofline study, with the layer / encoder / stock-torch context legs) under the key "c4"."""
    if args.workload != "c5":
        print(json.dumps(measure_single(args, args.workload, extras=True, with_cpu=True, dump_dir=args.dump_outputs)),
              flush=True)
        return
    line = measure_single(args, "c5", extras=False, with_cpu=False, dump_dir=args.dump_outputs)
    if not args.no_c4:
        c4 = measure_single(args, "c4", extras=True, with_cpu=True)
        line["cpu_baseline"] = c4.pop("cpu_baseline")          # bounded R-MAT sample: the same for both graphs
        line["layer"], line["encoder"] = c4.pop("layer"), c4.pop("encoder")
        for d in (line["layer"], line["encoder"]):
            if isinstance(d, dict):
                d["workload"] = c4["config"]["workload"]
        line["c4"] = {k: c4[k] for k in ("value", "unit", "ms_per_step", "config", "roofline", "roofline_bwd",
                                          "roofline_step", "e2e", "gpu_launches", "setup_s")}
    elif not args.no_cpu_baseline:
        eps, cms, cores = time_cpu_reference(2, 1, args.cpu_sample_nodes, args.cpu_sample_edges, 256)
        line["cpu_baseline"] = {"value": eps, "unit": "edges/s", "cores": cores, "kind": "port",
                                "sample": f"R-MAT {args.cpu_sample_nodes} nodes / {args.cpu_sample_edges} edges, F=256 "
                                          f"fp32, fwd+bwd, oracle port of torch_geometric propagate, {cms:.0f} ms/step"}
    if not args.no_small:
        # BASELINE.json configs[1] / configs[2]: encoder (and GAT layer) time on the reference's own dataset shapes
        for key in ("c2", "c3"):
            try:
                line[key] = measure_small(args, key, with_stock=not args.no_cpu_baseline)
            except Exception as ex:      # context legs never hide the headline
                line[key] = {"error": repr(ex)[:300]}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- our arm, N > 1 GPUs
FWD_VARIANTS = ("pull", "staged", "tma", "packed")
BWD_VARIANTS = ("push", "fetch", "fetch_barrier", "pipeline", "plain")


def run_partitioned(args):
    """bench.py --gpus N (N > 1): BASELINE.json configs[4] — the 10M-node / 200M-edge power-law graph,
    destination-row partitioned (gmlm_b200/partition.py), halo exchange + aggregation forward and backward.

    Transports (DESIGN.md §6).  forward: `pull` = one LDG pull kernel then the aggregation; `staged` = K LDG
    pull stages under the aggregation; `tma` = K stages moved by the bulk-copy engine (cp.async.bulk) from a
    few single-warp CTAs under the aggregation; `packed` = owner-side pack + copy-engine fetch per (owner,
    stage).  backward: `push` = owner slices stored into the owners' staging by the aggregation kernel;
    `fetch` = owner slices aggregated locally and fetched by copy engine behind pairwise signals;
    `fetch_barrier` = the same behind all-rank barriers; `pipeline`, `plain` = round-1 baselines.
    `--sweep` times every variant after ONE setup (per-variant ms to stderr and into the JSON line) and then
    times the full step with the fastest forward and backward."""
    import torch.distributed as dist

    import gmlm_b200 as G
    from gmlm_b200 import _lib, synth
    from gmlm_b200.partition import (PeerHalo, _pack, _unpack_add, build_local_part, cyclic_relabel,
                                     default_stage_fractions, halo_first_use_stage, partition_ranges,
                                     random_relabel, restage_part)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", str(rank)))
    if world == 1:
        raise SystemExit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    try:
        w = synth.WORKLOADS[args.workload]
        n = int(w.num_nodes * args.scale)
        e = int(w.num_edges * args.scale)
        feat = w.feat
        dtype = torch.bfloat16 if w.dtype == "bf16" else torch.float32
        esize = 2 if dtype == torch.bfloat16 else 4

        # every rank generates the same seeded graph (device RNG streams are identical across
        # identical GPUs) and keeps only its destination range
        t0 = time.perf_counter()
        ei = synth.make_graph(w, device=dev, num_nodes=n, num_edges=e)
        et = G.edge_type_from_degree(ei, n)                      # A2 needs the GLOBAL out-degree
        in_deg = torch.ops.gmlm.degree_i32(ei[1], n)
        if args.partition == "random":
            ei, ranges, _ = random_relabel(ei, n, world)         # balanced compute, ingress AND egress
        elif args.partition == "cyclic":
            ei, ranges, _ = cyclic_relabel(ei, n, world)
        else:
            # cost per node in edge units: fwd writes S (dst,rel) rows, bwd writes 1; each edge is read twice
            ranges = partition_ranges(in_deg, world, node_cost=2.5)
        live = sorted(torch.unique(et).tolist())                 # one relation->slot layout for all ranks
        part = build_local_part(ei, et, ranges, rank)
        del ei, et, in_deg
        torch.cuda.empty_cache()

        fwd_list = (args.sweep_fwd or list(FWD_VARIANTS)) if args.sweep else [args.fwd]
        bwd_list = [b for b in BWD_VARIANTS if b not in ("pipeline", "plain")] if args.sweep else [args.bwd]
        if args.halo == "nccl":
            fwd_list, bwd_list = ["nccl"], ["nccl"]
        if "packed" in fwd_list:
            # halo rows renumbered (owner, stage of first use, id): contiguous ranges for copy-engine transfers
            fr = default_stage_fractions(args.packed_stages)
            part = restage_part(part, halo_first_use_stage(part, live, fr), fr)
        g = G.RelGraph.build(part.edge_index, part.edge_type, part.n_local, 5, num_src=part.n_src, live_rels=live,
                             keep_seg=True)
        torch.cuda.synchronize()
        t_setup = time.perf_counter() - t0
        S = g.num_slots

        peer = None
        if args.halo == "p2p":
            peer = PeerHalo(part, feat, dtype)
            peer.build_backward_slices(g)
            if any(b in ("push", "fetch", "fetch_barrier") for b in bwd_list):
                peer.build_backward_push(g)
            if "packed" in fwd_list:
                peer.build_forward_packed(g)
            X, gX_buf = peer.X, peer.gX
        else:
            X = torch.empty((part.n_src, feat), dtype=dtype, device=dev)
            gX_buf = None
            n_send = int(sum(part.send_splits))
            send_buf = torch.empty((n_send, feat), dtype=dtype, device=dev)
            back_buf = torch.empty((n_send, feat), dtype=dtype, device=dev)
        # persistent buffers: the node features live in the head of the gather matrix X, the halo rows land
        # straight in its tail (no per-step concat / clone)
        X[: part.n_local] = synth.make_features(part.n_local, feat, device=dev, seed=42 + rank, dtype=dtype)
        x_local = X[: part.n_local]
        gh = synth.make_features(part.n_local * S, feat, device=dev, seed=7 + rank, dtype=dtype)
        h_buf = torch.empty((part.n_local * S, feat), dtype=dtype, device=dev)

        def _nk(csr):      # kernels of libgmlm_b200.so per aggregation call
            return 0 if csr is None else 1 + (2 if csr.n_hub else 0)

        staged_cache = {}

        def staged_plan(K):
            K = (K, args.stage_fractions)
            if staged_cache.get("K") != K:
                K = K[0]
                peer.build_forward_stages(g, n_stages=K, pull_ctas_overlapped=args.pull_ctas,
                                          fractions=default_stage_fractions(K, args.stage_fractions))
                staged_cache["K"] = (K, args.stage_fractions)
                staged_cache["nk"] = sum(_nk(st[0]) + (1 if st[3].numel() else 0) for st in peer.fwd_stages)

        def make_fwd(name):
            """-> (callable, launches per call, description)"""
            if name == "nccl":
                def f():
                    _pack(x_local, part.send_ids, out=send_buf)
                    dist.all_to_all_single(X[part.n_local:], send_buf, output_split_sizes=part.recv_splits,
                                           input_split_sizes=part.send_splits)
                    return G.spmm(X, g.fwd, _lib.AGG_MEAN, out=h_buf)
                return f, 1 + _nk(g.fwd), "pack kernel + NCCL all_to_all + aggregation"
            if name == "pull":
                def f():
                    peer.pull_forward()
                    return G.spmm(X, g.fwd, _lib.AGG_MEAN, out=h_buf)
                return f, 1 + _nk(g.fwd), "one LDG pull kernel over NVLink peer memory, then the aggregation"
            if name in ("staged", "tma"):
                K = args.fwd_stages
                staged_plan(K)
                tma = args.tma_ctas if name == "tma" else 0
                st0 = bool(args.tma_stage0) and tma > 0

                shape = tuple(args.tma_shape)

                def f():
                    peer.pull_tma_ctas, peer.pull_tma_stage0, peer.pull_tma_shape = tma, st0, shape
                    return peer.forward_staged(out=h_buf)
                what = (f"{K} halo stages by first use (block sizes '{args.stage_fractions}'); stage 0 by " +
                        ("bulk-copy (TMA) CTAs on every SM" if st0 else "the LDG pull kernel") + ", later stages " +
                        (f"by {tma} bulk-copy (TMA) CTAs (warps, ring KiB, rows per batch = {shape}; 0 = default)" if tma
                         else f"by {args.pull_ctas or 32} LDG CTAs") +
                        " under the aggregation blocks (two streams)")
                return f, staged_cache["nk"], what
            if name == "packed":
                def f():
                    return peer.forward_packed(out=h_buf)
                return f, sum(_nk(st[0]) for st in peer.packed_stages) + 1, \
                    f"owner-side pack + copy-engine fetch per (owner, stage), {args.packed_stages} stages"
            raise ValueError(name)

        def make_bwd(name):
            if name == "nccl":
                def f():
                    gX = G.spmm(gh, g.bwd, _lib.AGG_WEIGHTED)
                    dist.all_to_all_single(back_buf, gX[part.n_local:], output_split_sizes=part.send_splits,
                                           input_split_sizes=part.recv_splits)
                    gx = gX[: part.n_local]
                    off = 0
                    for cnt in part.send_splits:                 # peer order, unique ids per peer
                        if cnt:
                            _unpack_add(gx, part.send_ids[off:off + cnt], back_buf[off:off + cnt])
                        off += cnt
                    return gx
                return f, _nk(g.bwd) + world - 1, "aggregation + NCCL all_to_all + scatter-add per peer"
            sl = _nk(peer.slice_local) + sum(_nk(s_[0]) for s_ in peer.slices)
            if name == "push":
                return (lambda: peer.backward_pushed(gh)), sl + 1, \
                    "owner slices stored into the owners' staging by the aggregation kernel, local reduce"
            if name == "fetch":
                return (lambda: peer.backward_fetched(gh, local_last=True, signals=True)), sl + 1, \
                    "owner slices aggregated locally, fetched by copy engine behind pairwise signals, local rows last, one reduce"
            if name == "fetch_barrier":
                return (lambda: peer.backward_fetched(gh, local_last=False, signals=False)), sl + 1, \
                    "owner slices aggregated locally, fetched by copy engine behind all-rank barriers, one reduce"
            if name == "pipeline":
                return (lambda: peer.backward_pipelined(gh)), sl + world - 1, "owner slices pulled by copy engine + scatter-add"
            if name == "plain":
                def f():
                    G.spmm(gh, g.bwd, _lib.AGG_WEIGHTED, out=gX_buf)
                    return peer.pull_backward()
                return f, _nk(g.bwd) + 1, "whole transposed aggregation, then one pull-reduce kernel"
            raise ValueError(name)

        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def timed(fn, iters, warm=2):
            """mean ms per call, max over ranks (device time between barriers)."""
            for _ in range(warm):
                fn()
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            a.record()
            for _ in range(iters):
                fn()
            b.record()
            torch.cuda.synchronize()
            dist.barrier()
            t = torch.tensor([a.elapsed_time(b) / iters], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        sweep = None
        if args.sweep:
            sweep = {"forward_ms": {}, "backward_ms": {}}
            for name in fwd_list:
                if name in ("staged", "tma"):
                    for K in args.sweep_stages:
                        for c in (args.sweep_tma_ctas if name == "tma" else [0]):
                            for fr in args.sweep_fractions:
                                for s0 in (args.sweep_stage0 if name == "tma" else [0]):
                                    for shp in (args.sweep_tma_shapes if name == "tma" else ["0,0,0"]):
                                        args.fwd_stages, args.tma_ctas, args.stage_fractions, args.tma_stage0 = K, c, fr, s0
                                        args.tma_shape = [int(v) for v in shp.split(",")]
                                        fn, _, _ = make_fwd(name)
                                        key = f"{name}:K={K}:fr={fr}" + (f":ctas={c}:s0={s0}:shape={shp}" if name == "tma" else "")
                                        sweep["forward_ms"][key] = timed(fn, args.sweep_iters)
                                        if rank == 0:
                                            print(f"[sweep] fwd {key}: {sweep['forward_ms'][key]:.3f} ms", file=sys.stderr,
                                                  flush=True)
                else:
                    fn, _, _ = make_fwd(name)
                    sweep["forward_ms"][name] = timed(fn, args.sweep_iters)
                    if rank == 0:
                        print(f"[sweep] fwd {name}: {sweep['forward_ms'][name]:.3f} ms", file=sys.stderr, flush=True)
            if peer is not None and "tma" in fwd_list:
                # decomposition of the staged forward (measurement only): the pull chain alone, the blocks alone,
                # the blocks alone on ONE stream, and one whole-CSR aggregation
                sweep["decomposition_ms"] = {}
                fn, _, _ = make_fwd("tma")                     # the last swept configuration
                for tag, skip, ov in (("pulls_only", "agg", True), ("blocks_only_two_streams", "pull", True),
                                      ("blocks_only_one_stream", "pull", False)):
                    peer.debug_skip, peer.overlap_blocks = skip, ov
                    sweep["decomposition_ms"][tag] = timed(fn, args.sweep_iters)
                peer.debug_skip, peer.overlap_blocks = "", True
                sweep["decomposition_ms"]["whole_aggregation"] = timed(
                    lambda: G.spmm(X, g.fwd, _lib.AGG_MEAN, out=h_buf), args.sweep_iters)
                if rank == 0:
                    print(f"[sweep] decomposition {sweep['decomposition_ms']}", file=sys.stderr, flush=True)
            for name in bwd_list:
                fn, _, _ = make_bwd(name)
                sweep["backward_ms"][name] = timed(fn, args.sweep_iters)
                if rank == 0:
                    print(f"[sweep] bwd {name}: {sweep['backward_ms'][name]:.3f} ms", file=sys.stderr, flush=True)
            best_f = min(sweep["forward_ms"], key=sweep["forward_ms"].get)
            best_b = min(sweep["backward_ms"], key=sweep["backward_ms"].get)
            parts = best_f.split(":")
            args.fwd = parts[0]
            for kv in parts[1:]:
                k_, v_ = kv.split("=")
                if k_ == "K":
                    args.fwd_stages = int(v_)
                if k_ == "ctas":
                    args.tma_ctas = int(v_)
                if k_ == "fr":
                    args.stage_fractions = v_
                if k_ == "s0":
                    args.tma_stage0 = int(v_)
                if k_ == "shape":
                    args.tma_shape = [int(v) for v in v_.split(",")]
            args.bwd = best_b
            sweep["chosen"] = {"forward": best_f, "backward": best_b}

        fwd_name = "nccl" if args.halo == "nccl" else args.fwd
        bwd_name = "nccl" if args.halo == "nccl" else args.bwd
        fwd_fn, fwd_launches, fwd_what = make_fwd(fwd_name)
        bwd_fn, bwd_launches, bwd_what = make_bwd(bwd_name)
        launches_per_step = fwd_launches + bwd_launches

        PH = 2
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(PH + 1)] for _ in range(args.steps)]

        def step(k=None):
            if k is not None:
                ev[k][0].record()
            h = fwd_fn()                       # halo exchange + A5 on [local ‖ halo]
            if k is not None:
                ev[k][1].record()
            gx = bwd_fn()                      # A14 + halo-gradient return
            if k is not None:
                ev[k][2].record()
            return h, gx

        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sampler = None
        if rank == 0:
            sampler = ClockSampler(local_rank)
            sampler.start()
        a.record()
        for k in range(args.steps):
            step(k)
        b.record()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        timeline = None
        if peer is not None and fwd_name in ("staged", "tma"):   # one extra, untimed step with per-stage events
            peer.stage_timing = True
            step()
            torch.cuda.synchronize()
            peer.stage_timing = False
            timeline = {"pull_end_ms": peer.timeline_ms()[0], "block_end_ms": peer.timeline_ms()[1],
                        "rows_per_stage": peer.fwd_stage_rows}
            dist.barrier()
        phases = torch.tensor([statistics.mean(ev[k][i].elapsed_time(ev[k][i + 1]) for k in range(args.steps))
                               for i in range(PH)], device=dev, dtype=torch.float64)
        phases_all = [torch.zeros_like(phases) for _ in range(world)]
        dist.all_gather(phases_all, phases)
        ms = torch.tensor([a.elapsed_time(b) / args.steps], device=dev, dtype=torch.float64)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)               # device time, max over ranks
        # ---- e2e: every step each rank copies its node features from pinned host memory and reads a
        #      scalar of the result back (graph / CSR / halo plan stay resident: the graph is static).
        #      As in the 1-GPU arm, a copy stream lands step k+1's features in a staging buffer under step k's
        #      kernels; the step itself starts with a device copy staging -> x_local on the main stream, so the
        #      peers' view of x_local changes exactly where the unpipelined version changed it.
        x_host = x_local.cpu().pin_memory()
        e2e_steps = max(3, min(args.steps, 5))
        res_host = torch.empty(e2e_steps + 1, dtype=torch.float32).pin_memory()
        stage_bufs = [torch.empty_like(x_local), torch.empty_like(x_local)]
        copy_stream = torch.cuda.Stream()
        main_stream = torch.cuda.current_stream()
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        freed = [torch.cuda.Event(), torch.cuda.Event()]

        def issue_copy(k):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[k % 2])
                stage_bufs[k % 2].copy_(x_host, non_blocking=True)
                ready[k % 2].record(copy_stream)

        def e2e_run(steps):
            for ev_ in freed:
                ev_.record(main_stream)
            issue_copy(0)
            for k in range(steps):
                if k + 1 < steps:
                    issue_copy(k + 1)
                main_stream.wait_event(ready[k % 2])
                x_local.copy_(stage_bufs[k % 2])
                freed[k % 2].record(main_stream)
                _, gx_ = step()
                res_host[k:k + 1].copy_(gx_[:: max(1, part.n_local // 4096)].float().sum().reshape(1),
                                        non_blocking=True)

        e2e_run(1)
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        a.record()
        e2e_run(e2e_steps)
        b.record()
        torch.cuda.synchronize()
        dist.barrier()
        e2e_ms = torch.tensor([a.elapsed_time(b) / e2e_steps], device=dev, dtype=torch.float64)
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
        h2d = torch.tensor([float(x_host.numel() * esize)], device=dev, dtype=torch.float64)
        dist.all_reduce(h2d, op=dist.ReduceOp.SUM)
        halo_rows = torch.tensor([float(part.n_halo), float(part.edge_index.size(1)), float(part.n_local)],
                                 device=dev, dtype=torch.float64)
        halo_all = [torch.zeros_like(halo_rows) for _ in range(world)]
        dist.all_gather(halo_all, halo_rows)
        if rank == 0:
            clocks = sampler.stop()
            ms_step = float(ms.item())
            value = e / (ms_step * 1e-3)
            peak, peak_src = peaks()
            max_halo = max(float(t[0]) for t in halo_all)
            max_edges = max(float(t[1]) for t in halo_all)
            max_rows = max(float(t[2]) for t in halo_all)
            fwd_b, bwd_b = algorithmic_bytes(int(max_rows), int(max_edges), feat, esize, S)
            t_hbm = (fwd_b + bwd_b) / (peak * 1e9)
            t_link = 2 * max_halo * feat * esize / (NVLINK_GBS * 1e9)        # fwd + bwd exchange
            # compute and exchange can overlap: the bound is the slower of the two, per GPU
            roof_t = max(t_hbm, t_link)
            line = {
                "metric": "message-passing edges/sec fwd+bwd", "value": value, "unit": "edges/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": w.dtype, "data": "synthetic",
                "config": {"workload": w.title, "num_nodes": n, "num_edges": e, "feat": feat,
                           "parallelism": f"dst-row partition x{world} ({args.partition} ownership)",
                           "halo_forward": fwd_what, "halo_backward": bwd_what,
                           "l2": "inputs exceed L2", "halo_rows_per_rank": [int(t[0]) for t in halo_all],
                           "edges_per_rank": [int(t[1]) for t in halo_all],
                           "rows_per_rank": [int(t[2]) for t in halo_all]},
                "roofline": {"bound": "nvlink" if t_link > t_hbm else "hbm", "achieved": roof_t / (ms_step * 1e-3),
                             "peak": 1.0, "unit": "fraction of max(HBM, NVLink) time", "frac": roof_t / (ms_step * 1e-3),
                             "t_hbm_ms": t_hbm * 1e3, "t_nvlink_ms": t_link * 1e3, "traffic": None,
                             "peak_source": peak_src + f"; NVLink {NVLINK_GBS} GB/s per direction (B200_PROFILING.md)"},
                "cpu_baseline": None,
                "e2e": {"value": e / (float(e2e_ms.item()) * 1e-3), "unit": "edges/s",
                        "h2d_bytes_per_step": int(h2d.item()), "d2h_bytes_per_step": 4 * world,
                        "ms_per_step": float(e2e_ms.item()),
                        "note": "each rank copies its node features from pinned host memory every step "
                                "(double-buffered on a copy stream, then one device copy into the symmetric "
                                "x_local) and reads a scalar back; PCIe-bound"},
                "gpu_launches": launches_per_step * args.steps,
                "clocks": clocks, "setup_s": t_setup, "fwd_timeline_rank0": timeline, "sweep": sweep,
                "phases_ms_per_rank": {"order": ["forward (halo + aggregate)", "backward (aggregate + halo return)"],
                                       "ranks": [[round(float(v), 3) for v in t] for t in phases_all]},
            }
            print(json.dumps(line), flush=True)
    finally:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (development only)")
    ap.add_argument("--halo", default="p2p", choices=["p2p", "nccl"], help="N>1: halo exchange implementation")
    # defaults = the fastest variants of the round-2 sweeps on 8 GPUs (profiles/r2_scale_sweeps.md)
    ap.add_argument("--bwd", default="fetch", choices=list(BWD_VARIANTS), help="N>1: halo-gradient return (see run_partitioned)")
    ap.add_argument("--fwd", default="tma", choices=list(FWD_VARIANTS), help="N>1: forward halo transport (see run_partitioned)")
    ap.add_argument("--fwd-stages", type=int, default=6, help="N>1, --fwd staged|tma: halo stages (by first use)")
    ap.add_argument("--packed-stages", type=int, default=4, help="N>1, --fwd packed: stages")
    ap.add_argument("--tma-ctas", type=int, default=64, help="N>1, --fwd tma: bulk-copy CTAs per overlapped stage")
    ap.add_argument("--tma-stage0", type=int, default=0, help="N>1, --fwd tma: 1 = stage 0 by bulk copy too (one CTA per SM)")
    ap.add_argument("--pull-ctas", type=int, default=0, help="N>1, --fwd staged: CTA cap of the overlapped LDG pull kernels (0 = 32 CTAs of 1024 threads)")
    ap.add_argument("--sweep", action="store_true", help="N>1: time every transport variant after one setup, then the full step with the fastest")
    ap.add_argument("--sweep-iters", type=int, default=6)
    ap.add_argument("--sweep-stages", type=int, nargs="+", default=[4, 8])
    ap.add_argument("--sweep-tma-ctas", type=int, nargs="+", default=[16, 32, 64])
    ap.add_argument("--sweep-fractions", nargs="+", default=["fib"])
    ap.add_argument("--sweep-tma-shapes", nargs="+", default=["0,0,0"], help="warps,ringKiB,rowsPerBatch per variant")
    ap.add_argument("--tma-shape", type=int, nargs=3, default=[0, 0, 0],
                    help="N>1, --fwd tma: warps per CTA, ring KiB per CTA, rows per batch of the overlapped pull (0 = default)")
    ap.add_argument("--sweep-stage0", type=int, nargs="+", default=[0])
    ap.add_argument("--sweep-fwd", nargs="+", default=None, help="restrict the forward variants of --sweep")
    ap.add_argument("--stage-fractions", default="lin", choices=["fib", "lin", "flat"],
                    help="N>1, --fwd staged|tma: relative sizes of the aggregation blocks")
    ap.add_argument("--partition", default="random", choices=["random", "cyclic", "range"],
                    help="N>1: node ownership")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="N=1 default run: skip the configs[3] roofline-study leg")
    ap.add_argument("--no-layer", action="store_true")
    ap.add_argument("--no-small", action="store_true", help="N=1 default run: skip the configs[1]/[2] (C2/C3) legs")
    ap.add_argument("--cpu-sample-nodes", type=int, default=100_000)
    ap.add_argument("--cpu-sample-edges", type=int, default=2_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="N=1: write the last timed step's outputs (h, grad_x) to DIR/<name>.npy, float32, a fixed "
                         "row sample when larger than %d MiB in all" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "ours" or max(args.gpus, world) > 1):
        ap.error("--dump-outputs needs --impl ours on one GPU")
    if args.workload is None:
        args.workload = "c5"          # same graph at every N: the driver's scaling ratio compares like with like
    if args.impl == "reference":
        run_reference(args)
        return
    if max(args.gpus, world) > 1:
        run_partitioned(args)
        return
    run_single(args)


if __name__ == "__main__":
    main()
