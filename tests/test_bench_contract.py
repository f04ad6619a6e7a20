"""bench.py's contract line, checked on CPU through the one arm that needs no GPU (`--impl reference`: the CPU
restatement timed on the host cores).  The GPU arm prints the same keys plus roofline / gpu_launches / clocks; its line is
checked in tests/test_gpu_bench.py."""
import json
import os
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "cpu_baseline", "e2e"}


def _run(args, env=None, timeout=600):
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                         timeout=timeout, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]                 # exactly ONE JSON line
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-seconds", "0.3"])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["unit"] == "TFLOP/s" and d["higher_is_better"] is True and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert cb["extrapolation"]["by"] == "flops" and "median of 1 after" in cb["sample"]      # --steps sets the timed steps


def test_reference_arm_thread_count_survives_torchrun_env():
    """torch.distributed.run exports OMP_NUM_THREADS=1 for nproc > 1: the CPU arm must still use (and REPORT) every core the
    BLAS can drive, so its value is comparable across N (VERDICT r01 weak #5)."""
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="8", LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT="29998")
    env.pop("OPENBLAS_NUM_THREADS", None)
    d = _run(["--impl", "reference", "--gpus", "8", "--steps", "1", "--warmup", "1", "--ref-seconds", "0.3"], env=env)
    from threadpoolctl import threadpool_info
    import numpy  # noqa: F401
    cap = max(i["num_threads"] for i in threadpool_info() if i.get("user_api") == "blas")     # this process: default = all cores
    assert d["cpu_baseline"]["cores"] == cap and d["cpu_baseline"]["host_cores"] == os.cpu_count()
    assert f"on {cap} threads" in d["cpu_baseline"]["sample"]


def test_both_arms_share_config_and_metric():
    import bench
    import argparse
    a = argparse.Namespace(size=16384, grid=2, workload="blockmatrix", dtype="f64")
    assert bench.workload_config(a, 8)["workload"] == bench.workload_config(a, 1)["workload"]
    assert bench.metric_name(a) == bench.METRIC


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun only rank 0 runs the CPU arm; the other ranks print nothing and exit 0."""
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1", MASTER_ADDR="127.0.0.1", MASTER_PORT="29999")
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300, env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_our_arm_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "1"], stdout=subprocess.PIPE,
                         stderr=subprocess.PIPE, text=True, timeout=300)
    assert out.returncode != 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_reference_arm_tallskinny_workload():
    d = _run(["--impl", "reference", "--workload", "tallskinny", "--steps", "1", "--warmup", "1", "--ref-seconds", "0.3"])
    assert "tall-skinny" in d["metric"] and "configs[3]" in d["config"]["workload"]
    assert d["value"] > 0 and "rows" in d["cpu_baseline"]["sample"] and d["cpu_baseline"]["f2j_single_thread"]["cores"] == 1


def test_bad_arguments_are_refused():
    """No timed steps, or a dump of the CPU arm (its sample depends on the host's speed), is a usage error."""
    for args in (["--impl", "reference", "--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        out = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                             text=True, timeout=300, cwd=ROOT)
        assert out.returncode == 2 and "error:" in out.stderr and not out.stdout, args
