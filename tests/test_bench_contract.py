"""CPU: the bench.py output contract -- the committed B200 lines under profiles/ carry every key the driver reads, and the
reference arm (which needs no GPU) prints exactly one JSON line with its own required keys."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config"}


def _baseline():
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(ROOT, "profiles", "r[12]_bench_n*.json"))))
def test_committed_bench_lines_follow_the_contract(path):
    with open(path) as f:
        lines = [l for l in f.read().splitlines() if l.strip()]
    d = json.loads(lines[-1])
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["higher_is_better"] is True and d["scaling"] in ("weak", "strong") and d["data"] == "synthetic"
    assert d["vs_baseline"] is None                       # BASELINE.md publishes no number for this metric on any hardware
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["n_gpus"] in (1, 2, 4, 8) and d["warmup"] >= 3
    assert abs(d["value"] * d["ms_per_step"] * 1e-3 - 1.0) < 0.02          # scans/s and ms per scan describe the same run
    e2e = d["e2e"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(e2e)
    assert e2e["h2d_bytes_per_step"] > 30000 * 16 and e2e["d2h_bytes_per_step"] > 0
    assert e2e["value"] != d["value"]
    assert d["gpu_launches"] > 0
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r)
    assert r["bound"] == "hbm" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    c = d["clocks"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(c)
    assert not any("slowdown" in x and "power" not in x for x in c["reasons"])
    if d["n_gpus"] == 1 and d.get("cpu_baseline"):
        assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])
    want = _baseline().get("metric")
    if isinstance(want, str):
        assert d["metric"].split(" (")[0] in want or want.split(" (")[0] in d["metric"]


def test_reference_arm_prints_one_contract_line(tmp_path):
    env = dict(os.environ, OMP_NUM_THREADS="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--workload", "tiny", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1                                  # the ikd-Tree's own printf chatter must not reach stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["steps"] == 2
    dumped = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert set(dumped) == {"x", "P", "nearest", "nearest_count", "selected"}
    assert all(a.dtype in (np.float32, np.float64) for a in dumped.values())
    assert dumped["x"].shape == (26,) and dumped["P"].shape == (23, 23) and dumped["nearest"].shape == (400, 5, 4)
