#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path: N x N dense fp64 multiply (BASELINE.json metric).

Workload (BASELINE.json configs[2], the configuration the targets are quoted on, and it fits one GPU):
16384 x 16384 fp64 BlockMatrix multiply on a 2x2 block grid, (m,k,n) = (2,2,2) => 8 block products of
8192^3 (`BlockMatrix.multiply(other: BlockMatrix)`, matrix/BlockMatrix.scala:149-186), synthetic
U[0,1) inputs from the on-device XORShift generator (MTUtils.randomBlockMatrix).  One step = one full
multiply.  The same problem runs at N = 1, 2, 4, 8 GPUs ("strong" scaling); blocks are placed by
MatrixElemOpPartitioner order mod N; tiles move over NVLink peer memory behind the C ABI (mb_matmul_blocked_dist,
csrc/dist.cu), with grouped NCCL send/recv only as the fallback transport (MARLIN_B200_TRANSPORT=nccl).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--size S]          (N>1: launched by torchrun)
  python bench.py --impl reference ...   CPU restatement of the reference path (oracle port) on host cores
  python bench.py --dump-outputs DIR ... also write the last timed step's product to DIR/C.npy (see dump_outputs)

Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# The CPU legs (cpu_baseline, --impl reference) time numpy/OpenBLAS dgemm on ALL host cores.  torch.distributed.run
# exports OMP_NUM_THREADS=1 when nproc > 1 and OpenBLAS reads its thread count when the library is loaded, so the
# request has to be in the environment BEFORE the first `import numpy` (this file imports numpy lazily, below this
# line); cpu_threads() re-applies it through threadpoolctl and reports the count OpenBLAS really uses.
HOST_CORES = os.cpu_count() or 1
os.environ["OPENBLAS_NUM_THREADS"] = str(HOST_CORES)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")     # one hardware queue per stream (see marlin_b200/__init__.py)

FP64_PEAK_TFLOPS_MEASURED = 37.1   # scripts/dmma_bench.cu on this pool's B200 (profiles/r01_probe_*): 148 SM x 64 DFMA/clk x 1.965 GHz
METRIC = "fp64 dense multiply throughput (2*N^3 flop), 16384x16384 BlockMatrix 2x2 grid"
METRIC_TALL = "fp64 tall-skinny multiply throughput (2*M*K*N flop), DenseVecMatrix 1048576x1024 x 1024x1024"
DUMP_MAX_DIM = 2048                # --dump-outputs: at most 2048 x 2048 fp64 = 32 MiB


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--size", type=int, default=16384)
    ap.add_argument("--grid", type=int, default=2)
    ap.add_argument("--dtype", default="f64", choices=["f64", "bf16"],
                    help="tile element type: f64 (headline, configs[1..2]) or bf16 (configs[4]: --size 65536 --grid 4 --dtype bf16)")
    ap.add_argument("--workload", default="blockmatrix", choices=["blockmatrix", "tallskinny"],
                    help="blockmatrix: BlockMatrix x BlockMatrix (configs[1,2,4]); tallskinny: configs[3], DenseVecMatrix "
                         "1048576x1024 row-sharded times a replicated 1024x1024 (DenseVecMatrix.multiply(B: BDM))")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-int8-split", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=3.0, help="target seconds per CPU sample step of the cpu_baseline leg")
    ap.add_argument("--ref-seconds", type=float, default=3.0, help="target seconds per step of --impl reference")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the product of the last one as DIR/C.npy (fp64, or fp32 for bf16 tiles); "
                         f"a product with more than {DUMP_MAX_DIM} rows or columns is written on a fixed seeded sample of them")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's product; --impl reference times a host-dependent sample of the workload")
    return args


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_threads():
    """Ask the BLAS behind numpy for every host core and return (threads it will really use, library description).
    OpenBLAS wheels are built with a compile-time thread cap (64 or 128), so the count can be below os.cpu_count()."""
    import numpy as np  # noqa: F401  (loads the BLAS)
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=HOST_CORES, user_api="blas")
        infos = [i for i in threadpool_info() if i.get("user_api") == "blas"]
        if infos:
            i = infos[0]
            return int(i.get("num_threads", 1)), f"{i.get('internal_api', 'blas')} {i.get('version', '')} ({i.get('threading_layer', 'pthreads')})"
    except Exception:
        pass
    return int(os.environ.get("OPENBLAS_NUM_THREADS", "1")), "blas (threadpoolctl unavailable: thread count is the requested one)"


def cpu_port_sample(size: int, grid: int, target_seconds: float, steps: int = 5, warmup: int = 1, tall: bool = False):
    """The reference algorithm on host cores (oracle port, numpy/OpenBLAS dgemm on all threads), on a BOUNDED
    sample of the workload: one of the (grid^3) block products A(0,0) * B(0,0)[:, :w], w chosen so a step takes
    about `target_seconds` — or, for the tall-skinny workload, a slice of the rows of one partition times the broadcast
    1024 x 1024 matrix (DenseVecMatrix.scala:1660-1680).  Median of `steps` timed steps after a warm-up.
    Returns a dict: value (TFLOP/s), threads (actually used), cores (host), sample, ms, extrapolation."""
    import numpy as np
    from oracle import reference_model as rm
    threads, blas = cpu_threads()
    bs = size // grid
    rng = np.random.default_rng(42)
    probe = 2048
    a = np.asfortranarray(rng.random((probe, probe)))
    b = np.asfortranarray(rng.random((probe, probe)))
    rm.block_multiply(a, b, "blas")
    best = 1e9
    for _ in range(3):
        t0 = time.perf_counter()
        rm.block_multiply(a, b, "blas")
        best = min(best, time.perf_counter() - t0)
    gf = 2.0 * probe ** 3 / best / 1e9
    if tall:
        kdim = 1024
        rows = int(target_seconds * gf * 1e9 / (2.0 * kdim * kdim))
        rows = max(4096, min(65536, (rows // 1024) * 1024))
        A = np.ascontiguousarray(rng.random((rows, kdim)))             # the partition's rows, row-major
        B = np.asfortranarray(rng.random((kdim, kdim)))
        times = []
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            rm.block_multiply(A, B, "blas")                            # rowsMat * B per partition
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
        sec = statistics.median(times)
        sample = (f"{rows} of the 1048576 rows times the 1024x1024 broadcast matrix, numpy/OpenBLAS dgemm on {threads} threads "
                  f"({HOST_CORES} host cores); median of {len(times)} after {warmup} warm-up")
        return {"value": 2.0 * rows * kdim * kdim / sec / 1e12, "threads": threads, "cores": HOST_CORES, "blas": blas, "sample": sample,
                "ms": sec * 1e3, "extrapolation": {"by": "flops", "sample_flops": 2.0 * rows * kdim * kdim,
                                                   "workload_flops": 2.0 * 1048576 * kdim * kdim}}
    w = int(target_seconds * gf * 1e9 / (2.0 * bs * bs))
    w = max(64, min(bs, (w // 64) * 64))
    A = np.asfortranarray(rng.random((bs, bs)))
    B = np.asfortranarray(rng.random((bs, w)))
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        C = rm.block_multiply(A, B, "blas")          # SubMatrix.multiply -> dgemm (SubMatrix.scala:87-91)
        if grid > 1:
            C = rm.block_add(C, C)                    # one reduceByKey add per partial (BlockMatrix.scala:177)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    sec = statistics.median(times)
    flops = 2.0 * bs * bs * w
    sample = (f"one block product A(0,0)[{bs}x{bs}] * B(0,0)[:, :{w}] + one partial add, numpy/OpenBLAS dgemm on {threads} threads "
              f"({HOST_CORES} host cores); median of {len(times)} after {warmup} warm-up; rate extrapolated to the whole multiply by flops")
    return {"value": flops / sec / 1e12, "threads": threads, "cores": HOST_CORES, "blas": blas, "sample": sample, "ms": sec * 1e3,
            "extrapolation": {"by": "flops", "sample_flops": flops, "workload_flops": 2.0 * size ** 3}}


def f2j_sample(n: int = 768):
    """netlib-java's default backend is F2J, pure Java (the reference's README.md:31 says that is what runs unless
    native BLAS is installed): the oracle's C restatement of that loop nest, one thread, no FMA, as its stand-in."""
    import numpy as np
    from oracle import reference_model as rm
    rng = np.random.default_rng(7)
    a, b = np.asfortranarray(rng.random((n, n))), np.asfortranarray(rng.random((n, n)))
    rm.block_multiply(a[:64, :64], b[:64, :64], "f2j")
    t0 = time.perf_counter()
    rm.block_multiply(a, b, "f2j")
    sec = time.perf_counter() - t0
    return {"value": 2.0 * n ** 3 / sec / 1e12, "unit": "TFLOP/s", "cores": 1,
            "sample": f"{n}^3 product through the reference-BLAS dgemm loop nest in C (-ffp-contract=off), the stand-in for F2J"}


def workload_config(args, ws: int) -> dict:
    """The `config` object of the JSON line — the same for our arm and the reference arm at a given N."""
    N, g = args.size, args.grid
    tall, bf16 = args.workload == "tallskinny", args.dtype == "bf16"
    par = {1: "1 GPU: all 8 block products local (one grouped launch), k-sum accumulated in registers",
           2: "2 GPUs: 4 products each, k-sum local; tiles pulled over NVLink peer memory",
           4: "4 GPUs: 2 products each (same C tile), k-sum local; tiles pulled over NVLink peer memory",
           8: "8 GPUs: 1 product each (RDD partition == GPU); A/B tiles pulled over NVLink peer memory (copy engines), the k=2 "
              "partials reduce-scattered between the two holders by the GEMM epilogues (two launches per step: the peer's halves "
              "are stored into its HBM first, the own halves add the received partial in the epilogue)"}
    workload = (f"{N}x{N} fp64 BlockMatrix multiply, {g}x{g} block grid, (m,k,n)=({g},{g},{g}) "
                f"[BASELINE.json configs[2]; also the 1-GPU target size]")
    if tall:
        workload = "DenseVecMatrix 1048576x1024 (row-sharded) x replicated 1024x1024, fp64 [BASELINE.json configs[3]]"
    elif bf16:
        workload = f"{N}x{N} bf16 BlockMatrix multiply, {g}x{g} block grid, fp32 accumulate / fp32 C tiles [BASELINE.json configs[4]]"
    elif (N, g) != (16384, 2):
        workload = f"{N}x{N} fp64 BlockMatrix multiply, {g}x{g} block grid"
    headline = not (tall or bf16 or (N, g) != (16384, 2))
    return {"workload": workload,
            "parallelism": par.get(ws, f"{ws} GPUs") if headline else f"{ws} GPU(s), one process each",
            "l2": "inputs (2 GiB per operand) are far larger than the 126 MB L2; no explicit flush",
            "inputs": "U[0,1) fp64 from the on-device XORShift generator (MTUtils.randomBlockMatrix, seeds 42/43)"}


def metric_name(args) -> str:
    N, g = args.size, args.grid
    if args.workload == "tallskinny":
        return METRIC_TALL
    if args.dtype == "bf16":
        return f"bf16 dense multiply throughput (2*N^3 flop), {N}x{N} BlockMatrix {g}x{g} grid"
    if (N, g) != (16384, 2):
        return f"fp64 dense multiply throughput (2*N^3 flop), {N}x{N} BlockMatrix {g}x{g} grid"
    return METRIC


def run_reference(args):
    """The reference's own CPU implementation of the path on the box's host cores.  The Scala/Spark/Breeze reference cannot
    run here (no JVM), so this is the oracle port (kind "port"): the same block algorithm with numpy/OpenBLAS dgemm standing
    in for Breeze -> netlib-java native BLAS, on every host core, one bounded sample of the workload per step.  Under
    torchrun only rank 0 works; the thread count is forced and REPORTED (torchrun exports OMP_NUM_THREADS=1)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    tall = args.workload == "tallskinny"
    r = cpu_port_sample(args.size, args.grid, args.ref_seconds, steps=args.steps, warmup=max(1, min(2, args.warmup)), tall=tall)
    tf = r["value"]
    line = {
        "impl": "reference", "metric": metric_name(args), "value": tf, "unit": "TFLOP/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": tf, "unit": "TFLOP/s", "cores": r["threads"], "host_cores": r["cores"], "kind": "port", "blas": r["blas"],
                         "sample": r["sample"], "extrapolation": r["extrapolation"], "f2j_single_thread": f2j_sample()},
        "e2e": {"value": tf, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference = CPU restatement (oracle port, OpenBLAS dgemm standing in for Breeze->netlib-java); the Scala/Spark "
                "reference itself cannot run here (no JVM); each step times a bounded sample of the workload (cpu_baseline.sample) "
                "and the rate is extrapolated by flops; ms_per_step is the sample's time, not the whole multiply's",
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        loaded = [s for s, p in zip(sm, pw) if p > 300] or sm
        return {"sm_mhz": statistics.median(loaded) if loaded else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------ parity (checker, not product)
def _tile(sub, torch):
    """Logical (rows x cols) torch view of a packed column-major SubMatrix buffer, as fp64."""
    t = sub.buf[: sub.rows * sub.cols].view(sub.cols, sub.rows).t()
    return t if t.dtype == torch.float64 else t.to(torch.float64)


def freivalds_blockmatrix(A, B, Cm, ws, tol, probes=3):
    """Freivalds check of C = A*B on the device, at any number of ranks: for `probes` random vectors v (the same on every
    rank), y = C v against z = A (B v), with every tile-times-vector product done by torch (cuBLAS dgemv — independent of
    this repository's kernels) on the rank that holds the tile and the pieces summed with all_reduce.  Inputs are U[0,1),
    so (|A||B||v|)_i = z_i and the scaled error is max_i |y - z|_i / z_i.  An error of relative size d in ONE element of
    C moves its row sum by about d / n: with n = 16384 and tol = 1e-10 anything beyond ~2e-6 in a single element fails,
    and a wrong / missing / misplaced tile fails by orders of magnitude."""
    import torch
    import torch.distributed as dist
    dev = torch.device("cuda", torch.cuda.current_device())
    M, K, N = A.numRows(), A.numCols(), B.numCols()
    ceil = lambda a, b: -(-a // b)
    bm, bk, bn = ceil(M, A.numBlksByRow()), ceil(K, A.numBlksByCol()), ceil(N, B.numBlksByCol())
    gen = torch.Generator(device=dev).manual_seed(20260922)
    worst = 0.0
    for _ in range(probes):
        v = torch.rand(N, generator=gen, device=dev, dtype=torch.float64)
        w = torch.zeros(K, device=dev, dtype=torch.float64)
        for b, s in B.blocks:
            w[b.row * bk: b.row * bk + s.rows] += _tile(s, torch) @ v[b.column * bn: b.column * bn + s.cols]
        if ws > 1:
            dist.all_reduce(w)
        z = torch.zeros(M, device=dev, dtype=torch.float64)
        for b, s in A.blocks:
            z[b.row * bm: b.row * bm + s.rows] += _tile(s, torch) @ w[b.column * bk: b.column * bk + s.cols]
        y = torch.zeros(M, device=dev, dtype=torch.float64)
        seen = torch.zeros(M, device=dev, dtype=torch.float64)
        for b, s in Cm.blocks:
            y[b.row * bm: b.row * bm + s.rows] += _tile(s, torch) @ v[b.column * bn: b.column * bn + s.cols]
            seen[b.row * bm: b.row * bm + s.rows] += s.cols
        if ws > 1:
            dist.all_reduce(z); dist.all_reduce(y); dist.all_reduce(seen)
        if not bool((seen == N).all()):
            return {"max_scaled_err": float("inf"), "tol": tol, "ok": False, "method": "coverage: some C tile is missing or duplicated"}
        worst = max(worst, float(((y - z).abs() / z).max().item()))
    return {"max_scaled_err": worst, "tol": tol, "ok": bool(worst <= tol), "probes": probes, "n_ranks": ws,
            "method": "Freivalds on device: C v vs A (B v), torch/cuBLAS dgemv per tile on its owner + all_reduce; max_i |y-z|_i / (|A||B||v|)_i"}


def freivalds_rows(A_rows, B, C_rows, ws, tol, probes=3):
    """The same for the row-sharded multiply C_rows = A_rows * B (every rank checks its own shard, worst over ranks)."""
    import torch
    import torch.distributed as dist
    dev = torch.device("cuda", torch.cuda.current_device())
    gen = torch.Generator(device=dev).manual_seed(20260922)
    rowmajor = lambda s: s.buf[: s.rows * s.cols].view(s.rows, s.cols)
    a, c, b = rowmajor(A_rows), rowmajor(C_rows), _tile(B, torch)
    worst = 0.0
    for _ in range(probes):
        v = torch.rand(b.shape[1], generator=gen, device=dev, dtype=torch.float64)
        z = a @ (b @ v)
        worst = max(worst, float(((c @ v - z).abs() / z).max().item()))
    t = torch.tensor([worst], device=dev, dtype=torch.float64)
    if ws > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    worst = float(t.item())
    return {"max_scaled_err": worst, "tol": tol, "ok": bool(worst <= tol), "probes": probes, "n_ranks": ws,
            "method": "Freivalds on device per row shard: C v vs A (B v) with torch/cuBLAS dgemv; max_i |y-z|_i / (|A||B||v|)_i, worst rank"}


def dump_indices(M: int, N: int):
    """The rows and columns of an M x N product that --dump-outputs writes: all of them up to DUMP_MAX_DIM, else a fixed
    seeded sample of DUMP_MAX_DIM, sorted."""
    import numpy as np
    rng = np.random.default_rng(20261017)
    return tuple(np.sort(rng.choice(n, DUMP_MAX_DIM, replace=False)) if n > DUMP_MAX_DIM else np.arange(n) for n in (M, N))


def dump_outputs(out_dir: Path, Cm, M: int, N: int, tall: bool, bf16: bool, ws: int, rank: int):
    """Write the product C (M x N) a caller of the timed path receives as out_dir/C.npy, restricted to dump_indices(M, N),
    so that two builds run with the same arguments (hence the same seeded inputs) can be compared element for element.
    Every rank copies the sampled elements of the C tiles / row shard it holds into a zero matrix and the pieces are
    summed onto rank 0 (each element of C is held by exactly one rank)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    rows, cols = dump_indices(M, N)
    dev = torch.device("cuda", torch.cuda.current_device())
    out = torch.zeros(len(rows), len(cols), dtype=torch.float32 if bf16 else torch.float64, device=dev)
    cidx = torch.from_numpy(cols).to(dev)
    if tall:
        ids = np.asarray(Cm.ids)
        if len(ids):
            order = np.argsort(ids, kind="stable")
            pos = np.minimum(np.searchsorted(ids[order], rows), len(ids) - 1)
            hit = ids[order][pos] == rows
            s = Cm.data
            shard = s.buf[: s.rows * s.cols].view(s.rows, s.cols)                 # row-major shard
            src = torch.from_numpy(order[pos[hit]]).to(dev)
            out[torch.from_numpy(np.nonzero(hit)[0]).to(dev)] = shard.index_select(0, src).index_select(1, cidx).to(out.dtype)
    else:
        bm, bn = -(-M // Cm.numBlksByRow()), -(-N // Cm.numBlksByCol())
        for b, s in Cm.blocks:
            ri = np.nonzero((rows >= b.row * bm) & (rows < b.row * bm + s.rows))[0]
            ci = np.nonzero((cols >= b.column * bn) & (cols < b.column * bn + s.cols))[0]
            if len(ri) and len(ci):
                tile = s.buf[: s.rows * s.cols].view(s.cols, s.rows).t()          # packed column-major tile
                piece = tile.index_select(0, torch.from_numpy(rows[ri] - b.row * bm).to(dev))
                piece = piece.index_select(1, torch.from_numpy(cols[ci] - b.column * bn).to(dev))
                out[ri[0]: ri[-1] + 1, ci[0]: ci[-1] + 1] = piece.to(out.dtype)
    if ws > 1:
        dist.all_reduce(out)
    if rank == 0:
        out_dir.mkdir(parents=True, exist_ok=True)
        np.save(out_dir / "C.npy", out.cpu().numpy())


# ------------------------------------------------------------------------------------------ the other BASELINE configs
def measure_extra(kind: str, ws: int, rank: int, local_rank: int):
    """One of BASELINE.json's other configurations, measured in the same run as the headline so that the driver's
    record carries it: 'cfg1' = configs[1] (4096^2 fp64, one block), 'cfg3' = configs[3] (1048576x1024 x 1024x1024 fp64,
    row-sharded), 'cfg4' = configs[4] (65536^2 bf16, 4x4 grid).  Device-timed like the headline (CUDA events, max over
    ranks, >= 3 warm-up steps, ~1 s timed region so the clock sampler sees it), with its own parity and clocks."""
    import math
    import torch
    import torch.distributed as dist
    import marlin_b200 as mb
    from marlin_b200 import _native as nat
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    if kind == "cfg1":
        N, g, dt, name = 4096, 1, nat.MB_F64, "4096x4096 fp64 dense multiply, single block [BASELINE.json configs[1]]"
        A = mb.MTUtils.randomBlockMatrix(None, N, N, g, g, seed=42)
        B = mb.MTUtils.randomBlockMatrix(None, N, N, g, g, seed=43)
        flops, active = 2.0 * N ** 3, 1
        peak, peak_src, tol = FP64_PEAK_TFLOPS_MEASURED, "measured fp64 DMMA issue peak (scripts/dmma_bench.cu)", 1e-10
        kernel = "gemm_f64_dmma_grouped_kernel (DMMA.8x8x4 + TMA)"
    elif kind == "cfg3":
        rows_total, kdim = 1048576, 1024
        name = "DenseVecMatrix 1048576x1024 (row-sharded) x replicated 1024x1024, fp64 [BASELINE.json configs[3]]"
        A = mb.MTUtils.randomDenVecMatrix(None, rows_total, kdim, numPartitions=ws, seed=42)
        B = mb.SubMatrix(mb.MTUtils.randomBlockMatrix(None, kdim, kdim, 1, 1, seed=43).toBreeze())
        flops, active = 2.0 * rows_total * kdim * kdim, ws
        peak, peak_src, tol = FP64_PEAK_TFLOPS_MEASURED, "measured fp64 DMMA issue peak (scripts/dmma_bench.cu)", 1e-10
        kernel = "gemm_f64_dmma_kernel<T,N> (row-major C = A*B as C^T = B^T*A^T; DMMA.8x8x4 + TMA)"
    elif kind == "cfg4":
        N, g, dt = 65536, 4, nat.MB_BF16
        name = "65536x65536 bf16 BlockMatrix multiply, 4x4 block grid, fp32 accumulate / fp32 C tiles [BASELINE.json configs[4]]"
        A = mb.MTUtils.randomBlockMatrix(None, N, N, g, g, seed=42, dtype=dt)
        B = mb.MTUtils.randomBlockMatrix(None, N, N, g, g, seed=43, dtype=dt)
        flops, active = 2.0 * N ** 3, ws
        peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        peak_src, tol = "MEASURED_PEAKS.json bf16_tflops_sustained (cuBLAS bf16, seconds-long loop; burst: %s)" % peaks.get("bf16_tflops"), 1e-4
        kernel = "gemm_bf16_tcgen05_kernel (tcgen05.mma kind::f16 + TMEM + TMA), K segments over kk in one launch per C tile"
    else:
        raise ValueError(kind)
    torch.cuda.synchronize()

    def sync():
        if ws > 1:
            dist.barrier()
        torch.cuda.synchronize()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    Cm = None
    for _ in range(3):
        del Cm
        Cm = A.multiply(B)
    sync()
    e0.record()
    del Cm
    Cm = A.multiply(B)
    e1.record()
    sync()
    est = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if ws > 1:
        dist.all_reduce(est, op=dist.ReduceOp.MAX)
    steps = int(min(200, max(3, math.ceil(1000.0 / max(float(est.item()), 1e-3)))))
    sync()
    e0.record()
    for _ in range(steps):
        del Cm
        Cm = A.multiply(B)
    e1.record()
    sync()
    t = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if ws > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    clocks = sampler.stop() if rank == 0 else None
    value = flops / (ms * 1e-3) / 1e12
    parity = freivalds_rows(A.data, B, Cm.data, ws, tol) if kind == "cfg3" else freivalds_blockmatrix(A, B, Cm, ws, tol)
    del Cm, A, B
    torch.cuda.empty_cache()
    return {"config": name, "metric": "dense multiply throughput (2*M*K*N flop)", "value": value, "unit": "TFLOP/s", "ms_per_step": ms,
            "steps": steps, "warmup": 4, "n_gpus": ws, "dtype": "bf16" if kind == "cfg4" else "f64",
            "roofline": {"bound": "tensor", "achieved": value / active, "peak": peak, "unit": "TFLOP/s", "frac": value / active / peak,
                         "kernel": kernel, "peak_source": peak_src, "gpus_doing_work": active}, "parity": parity, "clocks": clocks}


# ------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import marlin_b200 as mb
    from marlin_b200 import _native as nat, comm, profiling

    ws = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if ws != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={ws}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local_rank)
    if ws > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    rt = mb.Runtime.get()
    N, g = args.size, args.grid
    flops = 2.0 * N * N * N

    bf16 = args.dtype == "bf16"
    tall = args.workload == "tallskinny"
    if tall:
        rows_total, kdim = 1048576, 1024
        A = mb.MTUtils.randomDenVecMatrix(None, rows_total, kdim, numPartitions=ws, seed=42)
        Bsub = mb.MTUtils.randomBlockMatrix(None, kdim, kdim, 1, 1, seed=43)       # generated where block (0,0) lives ...
        Bfull = Bsub.toBreeze()                                                   # ... and replicated (sc.broadcast)
        B = mb.SubMatrix(Bfull)
        flops = 2.0 * rows_total * kdim * kdim
        args.no_int8_split = True
    else:
        A = mb.MTUtils.randomBlockMatrix(None, N, N, g, g, seed=42, dtype=nat.MB_BF16 if bf16 else nat.MB_F64)
        B = mb.MTUtils.randomBlockMatrix(None, N, N, g, g, seed=43, dtype=nat.MB_BF16 if bf16 else nat.MB_F64)
        if bf16:
            args.no_e2e = True
            args.no_int8_split = True
    torch.cuda.synchronize()

    def barrier():
        if ws > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        return A.multiply(B)                       # BlockMatrix.multiply(other: BlockMatrix) / DenseVecMatrix.multiply(B: BDM)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()           # nvidia-smi needs ~1 s to start sampling: start before warm-up, read only loaded samples
    for _ in range(args.warmup):
        Cm = step()
        del Cm
    barrier()
    profiling.enable(True)
    l0 = rt.launch_count()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    Cm = None
    for _ in range(args.steps):
        del Cm
        Cm = step()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    phases = profiling.collect()
    profiling.enable(False)
    launches = rt.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms_total], device="cuda", dtype=torch.float64)
    if ws > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = flops / (ms_step * 1e-3) / 1e12

    # dominant kernel: the DMMA GEMM.  Average launch duration from the CUDA events bracketing each launch on the
    # launching stream; algorithmic flops per launch = this rank's share of the 2*N^3 flops / its launches per step
    # (1 grouped launch when the rank holds whole kk-sums, else one launch per 8192^3 block product).
    bs = N // g
    if tall:
        local_products, gemm_ms, gemm_n = 1, ms_total, args.steps          # one GEMM per row shard per step, nothing else
        launches_per_step = 1
        flops_per_launch = flops / ws
    else:
        plan = comm.plan_multiply(g, g, g, ws, A.owner, B.owner)
        local_products = len(plan.products.get(rank, []))
        gemm_ms, gemm_n = phases.get("gemm", (0.0, 0))
        # kernels inside one timed "gemm" span: 1 at N = 1 (grouped launch); 2 where the k partials are reduce-scattered
        # between two holders (the peer's halves first, flags as stream memory operations between the launches)
        launches_per_step = max(1, gemm_n // max(1, args.steps), int(launches) // max(1, args.steps))
        flops_per_launch = local_products * 2.0 * bs ** 3 / launches_per_step
    gemm_avg_ms = gemm_ms / max(1, gemm_n)
    spans_per_step = max(1, gemm_n // max(1, args.steps)) if not tall else 1
    gemm_avg_ms = gemm_avg_ms * spans_per_step / launches_per_step           # per kernel launch
    achieved = flops_per_launch / (gemm_avg_ms * 1e-3) / 1e12 if gemm_n else None
    # DRAM traffic of that launch: ncu (--set full) measured dram read+write of ONE 8192^3 block product
    # (profiles/r01_ncu_gemm_f64_dmma.md, round-1 capture of the same kernel body; no round-2 capture exists);
    # a launch that covers several products is scaled by their count.
    traffic = None
    traffic_source = None
    summary = ROOT / "profiles" / "ncu_summary.json"
    if summary.exists() and not tall and (N, g) == (16384, 2):
        try:
            per_product = json.loads(summary.read_text()).get("gemm_f64_dmma", {}).get("dram_bytes_per_launch")
            traffic = per_product * local_products / launches_per_step if per_product else None
            traffic_source = ("scaled from the round-1 ncu --set full capture of one 8192^3 block product "
                              "(profiles/r01_ncu_gemm_f64_dmma.md); not re-captured for the grouped launch")
        except Exception:
            traffic = None
    peak, peak_src = FP64_PEAK_TFLOPS_MEASURED, None
    if bf16:
        try:
            peak = float(json.loads((ROOT / "MEASURED_PEAKS.json").read_text())["bf16_tflops_sustained"])
            peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (cuBLAS bf16, seconds-long loop)"
        except Exception:
            peak, peak_src = 1400.0, "fallback sustained bf16 figure of B200_PROFILING.md"
        traffic = None
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_source,
                "kernel": ("gemm_bf16_tcgen05_kernel<N,N> (tcgen05.mma kind::f16 + TMEM + TMA)" if bf16 else
                           ("gemm_f64_dmma_kernel<T,N> (row-major C = A*B as C^T = B^T*A^T)" if tall else
                            "gemm_f64_dmma_grouped_kernel (DMMA.8x8x4 + TMA; " +
                            ("one launch per step" if ws == 1 else
                             f"{launches_per_step} launch(es) per rank and step; launch_ms_avg = the CUDA-event span around them / their "
                             "count, so it also holds the stream memory operations of the exchange protocol and any wait for "
                             "tiles / the peer's partial") + ")")),
                "launch_ms_avg": gemm_avg_ms,
                "flops_per_launch": flops_per_launch, "launches_per_step": launches_per_step,
                "peak_source": peak_src or "measured fp64 DMMA issue peak on this pool's B200 (scripts/dmma_bench.cu, "
                               "profiles/r01_probe_dmma_peak_and_gemm_v1.log); MEASURED_PEAKS.json carries no fp64 entry; "
                               "cuBLAS dgemm on the same GPU measured 36.2 TFLOP/s"}

    # ---- e2e: HOST buffers in, HOST buffers out, every step ----
    # N = 1: the C-ABI entry a JVM-held BlockMatrix would bind (mb_matmul_blocked_host): pinned host tiles -> pipelined
    #        H2D / 8 DMMA products / D2H.   N > 1: mb_matmul_blocked_dist_host — host tiles spread over the ranks'
    #        PCIe links, NVLink pulls, products, checkerboard reduce, D2H into shared pinned C tiles.
    e2e = None
    e2e_cleanup = None
    if not args.no_e2e and tall:
        # every rank: its row shard as pinned row-major host rows -> mb_matmul_rowsharded_host (row chunks pipelined over
        # H2D / DMMA / D2H streams) -> pinned row-major result rows.  PCIe-bound by construction: 128 flop per byte moved.
        import ctypes as C
        nloc = A.data.rows
        host_a = torch.empty(nloc * kdim, dtype=torch.float64).pin_memory()
        host_a.copy_(A.data.buf[: nloc * kdim])
        host_b = torch.empty(kdim * kdim, dtype=torch.float64).pin_memory()
        host_b.copy_(B.buf[: kdim * kdim])
        host_c = torch.empty(nloc * kdim, dtype=torch.float64).pin_memory()
        torch.cuda.synchronize()
        h2d, d2h_box = (nloc * kdim + kdim * kdim) * 8, [nloc * kdim * 8]
        path = ("mb_matmul_rowsharded_host (C ABI): pinned row-major rows -> 256 MiB row chunks pipelined over H2D / DMMA / "
                "D2H streams -> pinned row-major rows, every step")

        def e2e_step():
            nat.check(rt.lib.mb_matmul_rowsharded_host(rt.ctx, C.c_void_p(host_a.data_ptr()), nloc, kdim,
                                                       C.c_void_p(host_b.data_ptr()), kdim, C.c_void_p(host_c.data_ptr())))
    elif not args.no_e2e:
        import ctypes as C
        d2h_box = [0]
        h2d = 0
        if ws == 1:
            own_a = [(b, s) for b, s in A.blocks]
            own_b = [(b, s) for b, s in B.blocks]
            pin = lambda s: torch.empty(s.rows * s.cols, dtype=torch.float64).pin_memory().copy_(s.buf[: s.rows * s.cols].cpu())
            host_a = [(b, pin(s), s.rows, s.cols) for b, s in own_a]
            host_b = [(b, pin(s), s.rows, s.cols) for b, s in own_b]
            h2d = sum(t_.numel() * 8 for _, t_, _, _ in host_a + host_b)
            bs_ = N // g
            ha = {(b.row, b.column): t_ for b, t_, _, _ in host_a}
            hb = {(b.row, b.column): t_ for b, t_, _, _ in host_b}
            hc = {(i, j): torch.empty(bs_ * bs_, dtype=torch.float64).pin_memory() for i in range(g) for j in range(g)}
            pa = (C.c_void_p * (g * g))(*[ha[(i, kk)].data_ptr() for i in range(g) for kk in range(g)])
            pb = (C.c_void_p * (g * g))(*[hb[(kk, j)].data_ptr() for kk in range(g) for j in range(g)])
            pc = (C.c_void_p * (g * g))(*[hc[(i, j)].data_ptr() for i in range(g) for j in range(g)])
            lens = (C.c_int32 * g)(*([bs_] * g))
            d2h_box[0] = g * g * bs_ * bs_ * 8
            path = "mb_matmul_blocked_host (C ABI): pinned host tiles -> pipelined H2D / DMMA products / D2H, every step"

            def e2e_step():
                nat.check(rt.lib.mb_matmul_blocked_host(rt.ctx, pa, pb, g, g, g, lens, lens, lens, pc))
        else:
            # N > 1: the C-ABI end-to-end entry (mb_matmul_blocked_dist_host).  Every input tile sits in pinned host memory on
            # ONE of the ranks that need it (mb_dist_host_homes spreads the uploads over the PCIe links), C tiles are shared
            # pinned host arrays that the ranks computing a tile fill together; every step uploads all of A and B and
            # downloads all of C.
            from marlin_b200 import peer
            from marlin_b200.utils.mt_utils import MTUtils, UniformGenerator
            mesh = peer.PeerMesh.get()
            if mesh is None:         # the same verdict on every rank (PeerMesh.get is collective): report, do not die
                args.no_e2e = True
                e2e = {"error": "mb_comm_init failed on this box (no CUDA IPC / peer access between the GPUs?): the C-ABI end-to-end "
                                "entry needs the peer-memory communicator; device-timed `value` above used the NCCL transport"}
            if mesh is not None:
                lib = rt.lib
                gk = g
                a_home = (C.c_int32 * (g * gk))()
                b_home = (C.c_int32 * (gk * g))()
                nat.check(lib.mb_dist_host_homes(g, gk, g, ws, a_home, b_home))
                prank, cown = mesh.plan(g, gk, g)
                bs_ = N // g
                seeds_a, seeds_b = MTUtils._partition_seeds(42, g * g), MTUtils._partition_seeds(43, g * g)
                keep = []

                def host_tile(seed):
                    blk = mb.SubMatrix.empty(bs_, bs_, nat.MB_F64)
                    MTUtils._fill(blk, seed, 0, UniformGenerator(0.0, 1.0), row_major=False)      # the same values A / B hold on the device
                    t_ = torch.empty(bs_ * bs_, dtype=torch.float64).pin_memory()
                    t_.copy_(blk.buf[: bs_ * bs_])
                    keep.append(t_)
                    return t_.data_ptr()

                pa = (C.c_void_p * (g * gk))(*[host_tile(seeds_a[t]) if a_home[t] == rank else None for t in range(g * gk)])
                pb = (C.c_void_p * (gk * g))(*[host_tile(seeds_b[t]) if b_home[t] == rank else None for t in range(gk * g)])
                torch.cuda.synchronize()
                my_c = sorted({s // gk for s in range(g * gk * g) if prank[s] == rank})
                box = [os.urandom(6).hex() if rank == 0 else None]
                dist.broadcast_object_list(box, src=0)
                pc = (C.c_void_p * (g * g))()
                shared = {}
                for t in my_c:
                    ptr = C.c_void_p()
                    nat.check(lib.mb_host_alloc_shared(f"{box[0]}_c{t}".encode(), bs_ * bs_ * 8, C.byref(ptr)))
                    shared[t] = ptr
                    pc[t] = ptr
                lens = (C.c_int32 * g)(*([bs_] * g))
                h2d = sum(bs_ * bs_ * 8 for t in range(g * gk) if a_home[t] == rank) + sum(bs_ * bs_ * 8 for t in range(gk * g) if b_home[t] == rank)
                # bytes this rank downloads: whole tiles it holds alone, half of the tiles it shares (checkerboard of sub-blocks)
                holders = {}
                for s_ in range(g * gk * g):
                    holders.setdefault(s_ // gk, set()).add(prank[s_])
                d2h_box[0] = sum(bs_ * bs_ * 8 // len(holders[t]) for t in my_c)
                path = ("mb_matmul_blocked_dist_host (C ABI): pinned host tiles -> banded H2D on the rank that homes a tile + NVLink pulls by "
                        "the others -> one grouped DMMA launch per rank (starts on the first bands, sub-blocks in wavefront order) -> "
                        "sub-blocks a peer reduces are pushed to it by copy engine and added in its epilogue (checkerboard) -> D2H "
                        "into shared pinned C tiles, every step")

                def e2e_step():
                    nat.check(lib.mb_matmul_blocked_dist_host(mesh.comm, pa, a_home, pb, b_home, g, gk, g, lens, lens, lens, pc))

                def e2e_cleanup():
                    """Unmap the shared C tiles and remove their /dev/shm names (every holder unlinks; the second unlink is a no-op)."""
                    for t, ptr in shared.items():
                        lib.mb_host_free_shared(f"{box[0]}_c{t}".encode(), ptr, bs_ * bs_ * 8, 1)
                    shared.clear()

                def e2e_check():
                    """The e2e result against the device-resident result of the same multiply (owner ranks, whole tiles)."""
                    Cdev = {(b.row, b.column): s_ for b, s_ in A.multiply(B).blocks}
                    torch.cuda.synchronize()
                    dist.barrier()
                    worst = torch.zeros(1, device="cuda", dtype=torch.float64)
                    for t in my_c:
                        i, j = divmod(t, g)
                        if (i, j) in Cdev:
                            host = np.ctypeslib.as_array(C.cast(shared[t], C.POINTER(C.c_double)), shape=(bs_ * bs_,))
                            d = (torch.from_numpy(host).to(rt.device) - Cdev[(i, j)].buf[: bs_ * bs_]).abs().max()
                            worst = torch.maximum(worst, d.reshape(1))
                    dist.all_reduce(worst, op=dist.ReduceOp.MAX)
                    return float(worst.item())

    if not args.no_e2e:
        e2e_steps = max(2, min(args.steps, 3))
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        e0.record()
        for _ in range(e2e_steps):
            e2e_step()
        e1.record()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        # the step ends with a host-side wait for the D2H stream, so take the larger of device events and host wall clock
        t = torch.tensor([max(e0.elapsed_time(e1), wall_ms)], device="cuda", dtype=torch.float64)
        bts = torch.tensor([float(h2d), float(d2h_box[0])], device="cuda", dtype=torch.float64)
        if ws > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(bts, op=dist.ReduceOp.SUM)
        e2e_ms = float(t.item()) / e2e_steps
        e2e = {"value": flops / (e2e_ms * 1e-3) / 1e12, "unit": "TFLOP/s", "h2d_bytes_per_step": int(bts[0].item()),
               "d2h_bytes_per_step": int(bts[1].item()), "ms_per_step": e2e_ms, "steps": e2e_steps, "path": path}
        if ws > 1 and not tall:
            e2e["max_abs_diff_vs_device_result"] = e2e_check()
            e2e["fraction_of_device_value"] = e2e["value"] / value
    if e2e_cleanup is not None:
        barrier()                      # nobody is still copying into a tile another rank is about to unmap
        e2e_cleanup()

    # ---- extra (not the headline): the same multiply with the block GEMMs on the int8 tensor cores ----
    int8_split = None
    if ws == 1 and not args.no_int8_split:
        try:
            slices = 5                                          # 8-bit digits x 5 planes = 38 bits, 15 int8 GEMMs
            Cn = A.multiply(B)                                  # native result, kept for the error check
            rt.set_fp64_mode("int8x8", slices)
            for _ in range(2):
                Cs = A.multiply(B)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(3):
                Cs = A.multiply(B)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 3
            rt.set_fp64_mode("native")
            errs = []
            for (bn, sn), (bs_, ss) in zip(Cn.blocks, Cs.blocks):
                a_, b_ = sn.buf[: sn.rows * sn.cols], ss.buf[: ss.rows * ss.cols]
                errs.append(((a_ - b_).abs() / a_.abs()).max().item())     # U[0,1) inputs: C_ij = (|A||B|)_ij
            int8_split = {"value": flops / (ms * 1e-3) / 1e12, "unit": "TFLOP/s (fp64-equivalent)", "ms_per_step": ms,
                          "digit_bits": 8, "digit_planes": slices, "int8_gemms_per_product": slices * (slices + 1) // 2,
                          "int8_tops": flops * (slices * (slices + 1) // 2) / (ms * 1e-3) / 1e12,
                          "max_err_vs_native_scaled_by_absA_absB": max(errs), "tolerance": 1e-10,
                          "kernel": "gemm_ozaki_i8_kernel (tcgen05.mma.kind::i8, TMEM int32 accumulators) + split kernels",
                          "note": "opt-in mode (mb_set_fp64_mode); the headline value above is native IEEE fp64 on DMMA"}
            del Cn, Cs
        except Exception as exc:        # never let the extra break the headline line
            rt.set_fp64_mode("native")
            int8_split = {"error": str(exc)[:200]}

    # ---- parity of the LAST timed result, on device, at every N (the checker is torch/cuBLAS dgemv, not this library) ----
    parity = None
    if not args.no_parity:
        tol = 1e-4 if bf16 else 1e-10
        if tall:
            parity = freivalds_rows(A.data, B, Cm.data, ws, tol)
        else:
            parity = freivalds_blockmatrix(A, B, Cm, ws, tol)
    if args.dump_outputs:
        dump_outputs(Path(args.dump_outputs), Cm, rows_total if tall else N, kdim if tall else N, tall, bf16, ws, rank)
    del Cm

    # ---- the other BASELINE configurations, in the same run (only next to the default headline workload) ----
    extra_configs = None
    if not args.no_extra_configs and not tall and not bf16 and (N, g) == (16384, 2):
        del A, B
        torch.cuda.empty_cache()
        extra_configs = {}
        for kind in ("cfg1", "cfg3", "cfg4"):
            try:
                extra_configs[kind] = measure_extra(kind, ws, rank, local_rank)
            except Exception as exc:            # never let an extra break the headline line
                extra_configs[kind] = {"error": str(exc)[:300]}

    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        r = cpu_port_sample(N, g, args.cpu_seconds, tall=tall)
        cpu_baseline = {"value": r["value"], "unit": "TFLOP/s", "cores": r["threads"], "host_cores": r["cores"], "kind": "port",
                        "blas": r["blas"], "sample": r["sample"], "extrapolation": r["extrapolation"],
                        "f2j_single_thread": f2j_sample()}
    if ws > 1:
        dist.barrier()            # the other ranks wait for rank 0's CPU leg before tearing NCCL down

    if rank == 0:
        line = {
            "metric": metric_name(args), "value": value, "unit": "TFLOP/s", "n_gpus": ws, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16" if bf16 else "f64",
            "data": "synthetic",
            "config": workload_config(args, ws),
            "roofline": roofline, "e2e": e2e, "parity": parity, "cpu_baseline": cpu_baseline, "gpu_launches": int(launches),
            "fp64_on_int8_tensor_cores": int8_split, "extra_configs": extra_configs,
            "clocks": clocks,
            "phases_ms_per_step": {k: v[0] / args.steps for k, v in phases.items()},
            "pct_of_tensor_peak": 100.0 * value / (peak * ws),
        }
        if parity is not None and not parity["ok"]:
            line["error"] = f"PARITY FAILED: scaled error {parity['max_scaled_err']:.3e} > {parity['tol']:.1e}; the timing above is of a wrong result"
            line["value"] = None
        print(json.dumps(line), flush=True)
    if ws > 1:
        dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        raise SystemExit(3)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
