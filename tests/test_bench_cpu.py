"""bench.py pieces that need no GPU: the reference arm (`--impl reference` times the oracle port of the
reference path on the host cores and prints the contract line) and the algorithmic-bytes definition of
SURVEY §8(d) that every roofline figure divides by."""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def _run(*args):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_contract():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample-nodes", "5000",
             "--cpu-sample-edges", "100000")
    assert r["impl"] == "reference" and r["value"] > 0 and r["unit"] == "edges/s"
    assert r["metric"] == "message-passing edges/sec fwd+bwd" and r["higher_is_better"] is True
    assert r["cpu_baseline"]["kind"] == "port" and r["cpu_baseline"]["cores"] >= 1
    assert r["cpu_baseline"]["value"] == r["value"]
    assert r["e2e"] == {"value": r["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "10M nodes" in r["config"]["workload"] and r["scaling"] == "strong"      # same config as our arm's default


def test_reference_arm_other_ranks_exit_silently(monkeypatch):
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_algorithmic_bytes_match_survey_8d():
    import bench
    fwd, bwd = bench.algorithmic_bytes(2_000_000, 40_000_000, 256, 2, 4)           # C4, bf16, 4 live relations
    assert abs(fwd / 1e9 - 24.77) < 0.01 and abs(bwd / 1e9 - 21.71) < 0.01          # SURVEY §8(d): 24.77 + 21.71 GB
    assert abs((fwd + bwd) / 40_000_000 - 1162) < 1                                 # 1162 B/edge
    fwd5, bwd5 = bench.algorithmic_bytes(10_000_000, 200_000_000, 256, 2, 4)        # C5
    assert abs((fwd5 + bwd5) / 1e9 - 232.4) < 0.1                                   # "232.4 GB" whole graph on 1 GPU


def test_dump_outputs_is_float32_bounded_and_samples_the_same_rows(tmp_path):
    """--dump-outputs: a large output is cut to a fixed row sample within the byte budget, a small one is kept
    whole, everything is float32, and a second dump of the same tensors is identical."""
    import numpy as np
    import torch
    import bench
    big = torch.randn(3_000_000, 8).bfloat16()                 # 96 MB as float32: over the budget
    small = torch.randn(100, 8)
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, {"h": big, "grad_x": small})
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["grad_x.npy", "h.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES + 4096
    h = np.load(tmp_path / "a" / "h.npy")
    assert h.dtype == np.float32 and 0 < h.shape[0] < big.shape[0] and h.shape[1] == 8
    assert np.array_equal(h, np.load(tmp_path / "b" / "h.npy"))
    for r in (h[0], h[-1]):                                    # whole rows of the output, not mixed values
        assert bool((big.float() == torch.from_numpy(r)).all(1).any())
    assert np.array_equal(np.load(tmp_path / "a" / "grad_x.npy"), small.numpy())
