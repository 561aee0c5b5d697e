"""Time the GMLM encoder on GAT layers (GraphEncoder(conv="gat", heads=8)) on the C3 shape (synth.WORKLOADS["c3"]:
Amazon-ratings-shaped, 24.5k nodes, 93k edges, 300 features, hidden_channels = 512, so the layers are 512 -> 4096
features wide): forward + backward under torch.amp.autocast, eager and replayed through GraphedEncoderStep, and the
stock-torch GAT encoder restatement (tests/gat_encoder_ref.py: oracle.EncoderRef on GATConvRef layers,
index_select / index_add_ edge softmax) on the same GPU in the same process.
The stock arm runs in fp32, because GATConvRef fails under autocast.  CUDA events after warm-up.  Prints one JSON line with the card name and its power limit.
``--edge-types on`` times the encoder whose layers attend over the degree-bucket edge types
(``GraphEncoder(..., gat_edge_types=True)``) instead; ``both`` times the two encoders, one after the other, in the
same process (keys ``eager_ms`` / ``cuda_graph_ms`` and ``typed_eager_ms`` / ``typed_cuda_graph_ms``).
``--no-stock`` skips the stock-torch arm.

    python tools/time_gat_encoder.py [--iters 20] [--warmup 5] [--edge-types off|on|both] [--no-stock]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch  # noqa: E402

import gmlm_b200 as G  # noqa: E402
from gmlm_b200 import synth  # noqa: E402
sys.path.insert(0, str(Path(__file__).resolve().parents[1] / "tests"))
from gat_encoder_ref import GATEncoderRef  # noqa: E402


def _gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
        return name, power
    except Exception as ex:                        # the figures stay; say why the card is unnamed
        return torch.cuda.get_device_name(), f"unknown ({type(ex).__name__})"


def _time(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--edge-types", default="off", choices=["off", "on", "both"])
    ap.add_argument("--no-stock", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    w = synth.WORKLOADS["c3"]
    ei = synth.make_graph(w, device=dev)
    x = synth.make_features(w.num_nodes, w.feat, device=dev)
    xg = x.detach().requires_grad_(True)
    heads, out_dim = 8, 768

    def eager_step(m):
        # the stock arm runs fp32: GATConvRef cannot run under autocast (index_add_ of fp32 messages into fp16 z)
        with torch.amp.autocast("cuda", enabled=not isinstance(m, GATEncoderRef)):
            y = m(xg, ei) if isinstance(m, GATEncoderRef) else m.get_graph_embeddings(xg, ei)
        y.backward(torch.ones_like(y))
        xg.grad = None
        m.zero_grad(set_to_none=True)

    res = {"what": "GMLM encoder on GAT layers, forward + backward under torch.amp.autocast",
           "workload": w.title, "num_nodes": w.num_nodes, "num_edges": w.num_edges, "feat": w.feat,
           "hidden_channels": w.hidden, "heads": heads, "out_dim": out_dim, "iters": args.iters,
           "warmup": args.warmup, "edge_types": args.edge_types}
    for typed in {"off": [False], "on": [True], "both": [False, True]}[args.edge_types]:
        torch.manual_seed(0)
        enc = G.GraphEncoder(w.feat, w.hidden, out_dim, dropout_rate=0.0, conv="gat", heads=heads,
                             gat_edge_types=typed).to(dev)
        res["layer_widths"] = enc.dims[1:]
        pre = "typed_" if typed else ""
        res[pre + "eager_ms"] = _time(lambda: eager_step(enc), args.warmup, args.iters)
        step = G.GraphedEncoderStep(enc, x, ei, autocast=True, x_requires_grad=True)
        res[pre + "cuda_graph_ms"] = _time(lambda: step(x), args.warmup, args.iters)
        del step, enc
    res["gpu"], res["power_limit"] = _gpu_info()
    res["torch"] = torch.__version__
    if args.no_stock:
        print(json.dumps(res), flush=True)
        return
    torch.manual_seed(0)
    ref = GATEncoderRef(w.feat, w.hidden, out_dim, heads=heads, dropout_rate=0.0, use_checkpoint=False).to(dev)
    res["stock_torch_ms"] = _time(lambda: eager_step(ref), max(2, args.warmup // 2), max(5, args.iters // 4))
    res["stock_torch_what"] = ("GATEncoderRef (oracle EncoderRef on GATConvRef layers): GATConvRef "
                               "(index_select / scatter_reduce / index_add_ "
                               "edge softmax), stock GraphNorm and fusion ops, fp32 (it does not run under autocast: "
                               "index_add_ of fp32 messages into its fp16 z)")
    if "eager_ms" in res:
        res["speedup_vs_stock_eager"] = res["stock_torch_ms"] / res["eager_ms"]
        res["speedup_vs_stock_cuda_graph"] = res["stock_torch_ms"] / res["cuda_graph_ms"]
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
