"""bench.py contract (the driver parses this line): one JSON line with the required keys, the
roofline and cpu_baseline objects, an e2e number that moves host buffers, and a reference arm."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]


def _run(*args):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def test_bench_line_contract(lib_built, tmp_path):
    r = _run("--scale", "0.02", "--steps", "3", "--warmup", "3", "--cpu-sample-nodes", "5000",
             "--cpu-sample-edges", "100000", "--dump-outputs", str(tmp_path))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert k in r, k
    assert r["n_gpus"] == 1 and r["steps"] == 3 and r["unit"] == "edges/s" and r["vs_baseline"] is None
    assert r["dtype"] == "bf16" and r["data"] == "synthetic" and "workload" in r["config"]
    roof = r["roofline"]
    assert roof["bound"] == "hbm" and roof["unit"] == "GB/s" and roof["achieved"] > 0
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9
    assert r["cpu_baseline"]["kind"] == "port" and r["cpu_baseline"]["cores"] >= 1 and r["cpu_baseline"]["value"] > 0
    e2e = r["e2e"]
    assert e2e["h2d_bytes_per_step"] > 0 and e2e["d2h_bytes_per_step"] > 0 and 0 < e2e["value"] < r["value"]
    assert r["gpu_launches"] >= 2 * r["steps"]
    assert r["value"] > 0 and r["ms_per_step"] > 0
    # N=1 default: the 10M/200M graph of the scaling study, with the 2M/40M roofline study riding along
    assert "10M nodes" in r["config"]["workload"]
    c4 = r["c4"]
    assert "2M nodes" in c4["config"]["workload"] and c4["value"] > 0 and c4["roofline"]["achieved"] > 0
    assert r["encoder"] is None or "ms_fwd_bwd" in r["encoder"] or "error" in r["encoder"]
    # --dump-outputs: the headline step's two outputs, float32, within 64 MB in all
    assert sorted(p.name for p in tmp_path.iterdir()) == ["grad_x.npy", "h.npy"]
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    h, gx = np.load(tmp_path / "h.npy"), np.load(tmp_path / "grad_x.npy")
    assert h.dtype == gx.dtype == np.float32 and h.shape[1] == gx.shape[1] == r["config"]["feat"]
    assert np.isfinite(h).all() and np.isfinite(gx).all() and np.abs(h).max() > 0 and np.abs(gx).max() > 0


def test_bench_dump_is_the_same_every_run(lib_built, tmp_path):
    """Same arguments -> same seeded inputs -> the same outputs, bit for bit (the aggregation kernels are
    deterministic), so dumps of two builds can be compared output for output."""
    args = ("--scale", "0.01", "--steps", "2", "--warmup", "3", "--no-c4", "--no-small", "--no-cpu-baseline")
    for d in ("a", "b"):
        _run(*args, "--dump-outputs", str(tmp_path / d))
    for name in ("h.npy", "grad_x.npy"):
        assert np.array_equal(np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)), name
