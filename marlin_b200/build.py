"""Build libmarlin_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension).

The library is plain CUDA C++ behind a C ABI (include/marlin_b200.h); Python loads it with ctypes.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
LIBDIR = PKG / "lib"
LIB = LIBDIR / "libmarlin_b200.so"

SOURCES = ["capi.cu", "gemm_f64.cu", "gemm_bf16.cu", "gemm_ozaki.cu", "elementwise.cu", "blas12.cu", "peer.cu", "dist.cu", "factor.cu", "sparse.cu", "hostlogic.cpp"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; marlin_b200 needs the CUDA toolkit to build its sm_100a kernels")
    return exe


def needs_build() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = list(CSRC.glob("*")) + [ROOT / "include" / "marlin_b200.h", Path(__file__)]
    return any(p.stat().st_mtime > t for p in deps)


def build_library(force: bool = False, verbose: bool = False) -> Path:
    """Compile every translation unit and link the shared library. Returns its path."""
    if not force and not needs_build():
        return LIB
    LIBDIR.mkdir(exist_ok=True)
    objdir = LIBDIR / "obj"
    objdir.mkdir(exist_ok=True)
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = objdir / (src.rsplit(".", 1)[0] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-x", "cu", "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(str(obj))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
    tmp = LIBDIR / "libmarlin_b200.so.tmp"
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(tmp), *objs,
            "-Xcompiler", "-fPIC", "-cudart", "static"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    path = build_library(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)
