"""Bit parity of the RGCN layers, and of the GAT, GCN and linear_nt paths that share their plumbing, between two
builds of the library.  ``dump`` imports ``gmlm_b200`` from one tree, runs seeded layers forward and backward, and
saves the output and every gradient; ``compare`` reports per tensor whether two dumps are bit-equal, and the cases
a build raised on (the second build may fail where the first computes; the first may not).  Run one process per
tree (the two packages register the same torch.ops namespace):

    python tools/rgcn_parity_vs_parent.py dump --tree . --out /tmp/this.pt
    python tools/rgcn_parity_vs_parent.py dump --tree ../parent --out /tmp/parent.pt
    python tools/rgcn_parity_vs_parent.py compare /tmp/this.pt /tmp/parent.pt

Cases: RGCNConv(Fi -> Fo in {64, 22}, 5 relations, 30 bases) in its three formulations, forced, on the C2-shaped graph
of ``synth.WORKLOADS`` (300 features) and on an R-MAT graph with hub rows (256 features: 512-byte bf16 rows, the
band-ordered hub path); each under the bf16 pipeline, autocast, fp32, fp32 with a bf16 output and with
``use_tcgen05 = False`` (fp32 and bf16 activations).  Segment-compact runs for 16-bit operands only.  Plus GATConv in
fp32 and under autocast and GCNConv on both graphs, and linear_nt over three and four sources."""
from __future__ import annotations

import argparse
import sys
from pathlib import Path

import torch

# mode: (activation dtype, layer out_dtype, autocast, use_tcgen05)
MODES = {
    "bf16": (torch.bfloat16, torch.bfloat16, False, True),
    "autocast": (torch.float32, None, True, True),
    "fp32": (torch.float32, None, False, True),
    "fp32_out_bf16": (torch.float32, torch.bfloat16, False, True),
    "stock_fp32": (torch.float32, None, False, False),
    "stock_bf16": (torch.bfloat16, torch.bfloat16, False, False),
}
FORMS = {
    "aggregate_first": ("rgcn_transform", dict(transform_first=False, segment_compact=False)),
    "transform_first": ("rgcn_transform_first", dict(transform_first=True, segment_compact=False)),
    "segment_compact": ("rgcn_segment_compact", dict(transform_first=False, segment_compact=True)),
}


def _randn(*shape, seed):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def _grads(out, named):
    d = {"out": out.detach()}
    for name, t in named:
        d[name + ".grad"] = t.grad
    return {k: v.detach().cpu() for k, v in d.items() if v is not None}


def dump(tree: str, out_path: str) -> None:
    sys.path.insert(0, str(Path(tree).resolve()))
    import gmlm_b200 as G
    import gmlm_b200.nn as gnn
    from gmlm_b200 import synth
    from gmlm_b200.ops import linear_nt
    print(f"gmlm_b200 from {Path(G.__file__).parent}", flush=True)

    ran = []
    for fn in ("rgcn_transform", "rgcn_transform_first", "rgcn_segment_compact"):
        f = getattr(gnn, fn)
        setattr(gnn, fn, (lambda f, fn: lambda *a, **k: (ran.append(fn), f(*a, **k))[1])(f, fn))

    dev = torch.device("cuda:0")
    c2 = synth.WORKLOADS["c2"]
    graphs = [("c2", synth.make_graph(c2, seed=42), c2.num_nodes, c2.feat),
              ("rmat", synth.rmat_edges(40_000, 300_000, seed=3), 40_000, 256)]
    res, errors = {}, {}
    for gname, ei, n, fi in graphs:
        ei = ei.to(dev)
        et = G.edge_type_from_degree(ei, n)
        graph = G.get_rel_graph(ei, et, n, 5)
        print(f"{gname}: {n} nodes, {ei.size(1)} edges, forward hub rows {graph.fwd.n_hub}", flush=True)
        x32 = _randn(n, fi, seed=1).to(dev)
        for fo in (64, 22):
            sd = {"weight": _randn(30, fi, fo, seed=2) * fi ** -0.5, "comp": _randn(5, 30, seed=3) * 0.2,
                  "root": _randn(fi, fo, seed=4) * fi ** -0.5, "bias": _randn(fo, seed=5) * 0.1}
            gout = _randn(n, fo, seed=6).to(dev)
            for form, (fn, attrs) in FORMS.items():
                for mode, (xdt, odt, autocast, tc) in MODES.items():
                    if form == "segment_compact" and not (tc and (autocast or xdt == torch.bfloat16)):
                        continue
                    conv = G.RGCNConv(fi, fo, 5, 30, out_dtype=odt)
                    conv.load_state_dict(sd)
                    conv = conv.to(dev)
                    conv.use_tcgen05 = tc
                    for k, v in attrs.items():
                        setattr(conv, k, v)
                    x = x32.to(xdt, copy=True).requires_grad_(True)
                    key = f"rgcn/{gname}/fo{fo}/{form}/{mode}"
                    ran.clear()
                    try:
                        with torch.amp.autocast("cuda", enabled=autocast):
                            y = conv(x, graph)
                        y.backward(gout.to(y.dtype))
                    except RuntimeError as e:
                        errors[key] = f"{type(e).__name__}: {str(e).splitlines()[0]}"
                        continue
                    assert ran == [fn], (form, mode, ran)
                    res[key] = _grads(y, [("x", x)] + list(conv.named_parameters()))
        for mode in ("fp32", "autocast"):
            torch.manual_seed(7)
            gat = G.GATConv(fi, 64, heads=2).to(dev)
            x = x32.clone().requires_grad_(True)
            with torch.amp.autocast("cuda", enabled=mode == "autocast"):
                y = gat(x, ei)
            y.backward(_randn(*y.shape, seed=8).to(dev))
            res[f"gat/{gname}/{mode}"] = _grads(y, [("x", x)] + list(gat.named_parameters()))
        torch.manual_seed(9)
        gcn = G.GCNConv(fi, 128).to(dev)
        x = x32.clone().requires_grad_(True)
        y = gcn(x, ei)
        y.backward(_randn(*y.shape, seed=10).to(dev))
        res[f"gcn/{gname}"] = _grads(y, [("x", x)] + list(gcn.named_parameters()))
    n = 30_000
    for widths in ((100, 60, 40), (64, 64, 128, 40)):
        xs = [_randn(n, w, seed=11 + i).to(dev).requires_grad_(True) for i, w in enumerate(widths)]
        wt = (_randn(96, sum(widths), seed=20) * 0.05).to(dev).requires_grad_(True)
        bias = (_randn(96, seed=21) * 0.1).to(dev).requires_grad_(True)
        y = linear_nt(xs, wt, bias, out_dtype=torch.float32)
        y.backward(_randn(n, 96, seed=22).to(dev))
        res[f"linear_nt/{len(widths)}_sources"] = _grads(y, [(f"x{i}", t) for i, t in enumerate(xs)] +
                                                         [("wt", wt), ("bias", bias)])
    torch.cuda.synchronize()
    torch.save({"cases": res, "errors": errors}, out_path)
    print(f"{len(res)} cases, {sum(len(v) for v in res.values())} tensors, {len(errors)} cases raised -> {out_path}",
          flush=True)


def compare(a_path: str, b_path: str) -> int:
    da, db = torch.load(a_path, weights_only=False), torch.load(b_path, weights_only=False)
    a, b = da["cases"], db["cases"]
    bad = 0
    for case, msg in sorted(da["errors"].items()):
        print(f"{case}: the first build raised {msg}")
        bad += 1
    for case, msg in sorted(db["errors"].items()):
        print(f"{case}: the second build raised {msg}" + ("; the first computed it" if case in a else ""))
    missing = (set(a) ^ set(b)) - set(db["errors"])
    if missing:
        print(f"case lists differ: {sorted(missing)}")
        bad += len(missing)
    for case in sorted(a.keys() & b.keys()):
        for name in sorted(a[case].keys() | b[case].keys()):
            ta, tb = a[case].get(name), b[case].get(name)
            if ta is None or tb is None or ta.dtype != tb.dtype or ta.shape != tb.shape:
                print(f"{case} {name}: missing or dtype / shape differs")
                bad += 1
                continue
            eq = torch.equal(ta, tb) and torch.equal(ta.isnan(), tb.isnan())
            diff = float((ta.double() - tb.double()).abs().nan_to_num(0.0).max()) if ta.numel() else 0.0
            print(f"{case} {name} {tuple(ta.shape)} {str(ta.dtype).replace('torch.', '')}: bit-equal={eq} "
                  f"max|diff|={diff:.3e}")
            bad += not eq
    print("ALL BIT-EQUAL" if bad == 0 else f"{bad} TENSORS DIFFER")
    return 1 if bad else 0


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    sub = ap.add_subparsers(dest="cmd", required=True)
    d = sub.add_parser("dump")
    d.add_argument("--tree", required=True, help="repository root whose gmlm_b200 is imported")
    d.add_argument("--out", required=True, help="file the tensors are saved to")
    c = sub.add_parser("compare")
    c.add_argument("a")
    c.add_argument("b")
    args = ap.parse_args()
    if args.cmd == "dump":
        dump(args.tree, args.out)
        return 0
    return compare(args.a, args.b)


if __name__ == "__main__":
    sys.exit(main())
