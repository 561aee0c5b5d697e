#!/usr/bin/env python
"""Development: GraphNorm(+GELU) forward/backward time at the encoder's widths, bf16 and fp32, then the
LayerNorm closing MultiScaleFusion against torch's.  Prints the device and its power limit first."""
import sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch
import gmlm_b200 as G
dev = torch.device("cuda:0")
try:
    import subprocess
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip())
except OSError:
    print(torch.cuda.get_device_name(dev))
m = 2_000_000
for dtype, c in ((torch.bfloat16, 64), (torch.bfloat16, 512), (torch.float32, 64), (torch.float32, 512)):
    norm = G.GraphNorm(c).to(dev)
    x = torch.randn(m, c, device=dev).to(dtype).requires_grad_(True)
    gy = torch.randn(m, c, device=dev).to(dtype)
    # the statistics pass alone (colstats: one read of x)
    for _ in range(3):
        torch.ops.gmlm.colstats(x)
    a, b = (torch.cuda.Event(enable_timing=True) for _ in range(2))
    a.record()
    for _ in range(20):
        torch.ops.gmlm.colstats(x)
    b.record(); torch.cuda.synchronize()
    st = a.elapsed_time(b) / 20
    for _ in range(2):
        y = norm(x, fuse_gelu=True); y.backward(gy); x.grad = None
    torch.cuda.synchronize()
    a, b, c_ = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    f = bw = 0.0
    for _ in range(5):
        a.record(); y = norm(x, fuse_gelu=True); b.record(); y.backward(gy); c_.record(); torch.cuda.synchronize()
        f += a.elapsed_time(b); bw += b.elapsed_time(c_); x.grad = None
    gb = m * c * x.element_size() / 1e9
    print(f"{str(dtype)[6:]} C={c}: colstats {st:.3f} ms ({gb/st*1e3:.0f} GB/s)  fwd {f/5:.3f} ms ({3*gb/(f/5)*1e3:.0f} GB/s of 3 passes)  bwd {bw/5:.3f} ms ({5*gb/(bw/5)*1e3:.0f} GB/s of 5 passes)")

# LayerNorm closing MultiScaleFusion: [2M, 768] bf16, ours vs torch
c = 768
w = torch.ones(c, device=dev, requires_grad=True); b = torch.zeros(c, device=dev, requires_grad=True)
x = torch.randn(m, c, device=dev).bfloat16().requires_grad_(True)
gy = torch.randn(m, c, device=dev).bfloat16()
tl = torch.nn.LayerNorm(c).to(dev).bfloat16()
for name, fn in (("ours", lambda: G.layer_norm(x, w, b, 1e-5)), ("torch", lambda: tl(x))):
    for _ in range(2):
        fn().backward(gy); x.grad = None
    torch.cuda.synchronize()
    a, bb, c_ = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    f = bw = 0.0
    for _ in range(5):
        a.record(); y = fn(); bb.record(); y.backward(gy); c_.record(); torch.cuda.synchronize()
        f += a.elapsed_time(bb); bw += bb.elapsed_time(c_); x.grad = None
    gb = m * c * 2 / 1e9
    print(f"LayerNorm {name}: fwd {f/5:.3f} ms ({2*gb/(f/5)*1e3:.0f} GB/s)  bwd {bw/5:.3f} ms ({3*gb/(bw/5)*1e3:.0f} GB/s)")
