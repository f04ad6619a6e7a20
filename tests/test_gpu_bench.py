"""bench.py's GPU arm on a small configuration (BASELINE configs[1]: 4096^2 fp64, one block): the one JSON line carries
every key of the contract, device-timed throughput is plausible, and the e2e leg really moves the operands."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]


def test_gpu_arm_line_small_config():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--size", "4096", "--grid", "1", "--steps", "3", "--warmup", "3",
                          "--no-cpu-baseline", "--no-int8-split"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks"):
        assert key in d, key
    assert d["unit"] == "TFLOP/s" and d["dtype"] == "f64" and d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 3
    assert 5.0 < d["value"] < 40.0                                   # fp64 tensor peak is 37.1 TFLOP/s
    assert abs(d["value"] - 2 * 4096 ** 3 / (d["ms_per_step"] * 1e-3) / 1e12) < 1e-6 * d["value"]
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and 0.1 < r["frac"] <= 1.0 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 2 * 4096 * 4096 * 8 and e["d2h_bytes_per_step"] == 4096 * 4096 * 8
    assert 0 < e["value"] < d["value"]                               # host buffers in and out cannot beat the resident number
    assert d["gpu_launches"] >= 3
    assert "sm_mhz" in d["clocks"] and "reasons" in d["clocks"]


def test_dump_outputs_is_the_last_product(oracle, tmp_path):
    """--dump-outputs writes C = A*B of the timed path on the rows and columns bench.dump_indices samples (2100 > 2048:
    the sampled case), the inputs being the seeded generator streams the oracle restates."""
    import bench
    n = 2100
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--size", str(n), "--grid", "2", "--steps", "2", "--warmup", "1",
                          "--no-cpu-baseline", "--no-int8-split", "--no-e2e", "--dump-outputs", str(tmp_path)],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    assert json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])["steps"] == 2
    assert sorted(p.name for p in tmp_path.iterdir()) == ["C.npy"]
    got = np.load(tmp_path / "C.npy")
    r, c = bench.dump_indices(n, n)
    A = oracle.random_block_matrix(n, n, 2, 2, seed=42).to_breeze()
    B = oracle.random_block_matrix(n, n, 2, 2, seed=43).to_breeze()
    want = A[r] @ B[:, c]                                            # U[0,1) inputs: |A||B| = A B
    assert got.dtype == np.float64 and got.shape == (bench.DUMP_MAX_DIM, bench.DUMP_MAX_DIM)
    assert (np.abs(got - want) / want).max() <= 1e-10
