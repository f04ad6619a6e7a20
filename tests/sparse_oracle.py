"""CPU oracle of the sparse block path: the C restatements in tests/sparse_oracle.c (built with gcc -ffp-contract=off into
a temporary directory on first use) and a model of BlockMatrix.multiply over grids whose blocks may be sparse.

A sparse block is a `Csc` (rows, cols, col_ptr, row_idx, val); a dense block is a 2-D float64 ndarray.  Paths cited are
relative to the reference's src/main/scala/edu/nju/pasalab/marlin/."""
from __future__ import annotations

import atexit
import ctypes as C
import shutil
import subprocess
import tempfile
from pathlib import Path
from typing import Dict, NamedTuple, Tuple

import numpy as np

_SRC = Path(__file__).resolve().parent / "sparse_oracle.c"
_lib = None

_IP = C.POINTER(C.c_int32)
_DP = C.POINTER(C.c_double)


class Csc(NamedTuple):
    rows: int
    cols: int
    col_ptr: np.ndarray     # int32[cols+1]
    row_idx: np.ndarray     # int32[nnz]
    val: np.ndarray         # float64[nnz]

    @staticmethod
    def from_columns(rows: int, cols, columns) -> "Csc":
        """One (indices, values) pair or None per column, like the reference's Array[SparseVector]."""
        cp, ri, v = [0], [], []
        for col in columns:
            if col is not None:
                ri.extend(col[0]); v.extend(col[1])
            cp.append(len(ri))
        return Csc(rows, cols, np.array(cp, np.int32), np.array(ri, np.int32), np.array(v, np.float64))

    @staticmethod
    def from_dense(a: np.ndarray) -> "Csc":
        """The stored entries are the nonzeros of `a` (a -0.0 is not stored)."""
        import scipy.sparse as sps
        m = sps.csc_matrix(np.asarray(a))
        m.sort_indices()
        return Csc(a.shape[0], a.shape[1], m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data.astype(np.float64))


def _load() -> C.CDLL:
    global _lib
    if _lib is None:
        d = Path(tempfile.mkdtemp(prefix="marlin_sparse_oracle_"))
        atexit.register(shutil.rmtree, d, True)
        so = d / "libsparse_oracle.so"
        subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-Wall", "-ffp-contract=off", "-fno-fast-math", "-o",
                        str(so), str(_SRC)], check=True)
        _lib = C.CDLL(str(so))
        _lib.sp_mult_sparse_dense.restype = C.c_int
    return _lib


def _p(a, t):
    return a.ctypes.data_as(t)


def _csc_args(s: Csc):
    cp = np.ascontiguousarray(s.col_ptr, np.int32)
    ri = np.ascontiguousarray(s.row_idx, np.int32) if s.row_idx.size else np.zeros(1, np.int32)
    v = np.ascontiguousarray(s.val, np.float64) if s.val.size else np.zeros(1)
    return cp, ri, v


def mult_dense_sparse(a: np.ndarray, b: Csc) -> np.ndarray:
    """LibMatrixMult.scala:15-41"""
    assert a.shape[1] == b.rows
    a = np.asfortranarray(a, dtype=np.float64)
    m, n = a.shape[0], b.cols
    c = np.zeros((m, n), order="F")
    cp, ri, v = _csc_args(b)
    _load().sp_mult_dense_sparse(m, n, _p(a, _DP), max(1, m), _p(cp, _IP), _p(ri, _IP), _p(v, _DP), _p(c, _DP))
    return c


def mult_sparse_dense(a: Csc, b: np.ndarray, literal: bool = False):
    """LibMatrixMult.scala:43-77.  literal=False: as defined (k ascending).  literal=True: the reference's loop as written
    (`bixi = i * cd + bi`, :60); returns None when that loop would read past the end of B."""
    assert a.cols == b.shape[0]
    b = np.asfortranarray(b, dtype=np.float64)
    m, K, n = a.rows, a.cols, b.shape[1]
    c = np.zeros((m, n), order="F")
    cp, ri, v = _csc_args(a)
    rc = _load().sp_mult_sparse_dense(m, K, n, _p(cp, _IP), _p(ri, _IP), _p(v, _DP), _p(b, _DP) if b.size else None,
                                      _p(c, _DP), 0 if literal else 1)
    return None if rc != 0 else c


def multiply(a: Csc, b: Csc) -> np.ndarray:
    """SparseMatrix.multiply (Matrices.scala:208-231)"""
    assert a.cols == b.rows
    c = np.zeros((a.rows, b.cols), order="F")
    acp, ari, av = _csc_args(a)
    bcp, bri, bv = _csc_args(b)
    _load().sp_multiply(a.rows, b.cols, _p(acp, _IP), _p(ari, _IP), _p(av, _DP), _p(bcp, _IP), _p(bri, _IP), _p(bv, _DP),
                        _p(c, _DP))
    return c


def to_dense(a: Csc) -> np.ndarray:
    """SparseMatrix.toDense (Matrices.scala:185-198)"""
    c = np.zeros((a.rows, a.cols), order="F")
    cp, ri, v = _csc_args(a)
    _load().sp_to_dense(a.rows, a.cols, _p(cp, _IP), _p(ri, _IP), _p(v, _DP), _p(c, _DP))
    return c


def rand_count(rows: int, cols: int, sparsity: float) -> int:
    """(numCols * sparsity).toInt (Matrices.scala:240), with the product's refusals."""
    if not sparsity >= 0:
        raise ValueError("sparsity must be >= 0")
    s = int(float(cols) * float(sparsity))
    if s > rows or s * cols >= 2 ** 31:
        raise ValueError(f"{s} rows per column from {rows} rows")
    return s


def rand(rows: int, cols: int, sparsity: float, seed: int) -> Csc:
    """The product's seeded SparseMatrix.rand."""
    count = rand_count(rows, cols, sparsity)
    cp = np.zeros(cols + 1, np.int32)
    ri = np.zeros(max(1, count * cols), np.int32)
    v = np.zeros(max(1, count * cols))
    _load().sp_rand(rows, cols, count, C.c_int64(seed), _p(cp, _IP), _p(ri, _IP), _p(v, _DP))
    return Csc(rows, cols, cp, ri[:count * cols], v[:count * cols])


def block_product(a, b) -> np.ndarray:
    """SubMatrix.multiply (SubMatrix.scala:87-105) for a product with at least one sparse operand."""
    if isinstance(a, Csc) and isinstance(b, Csc):
        return multiply(a, b)
    if isinstance(b, Csc):
        return mult_dense_sparse(a, b)
    if isinstance(a, Csc):
        return mult_sparse_dense(a, b)
    raise ValueError("dense x dense products are the DMMA path, not modelled here")


def block_multiply(a_blocks: Dict[Tuple[int, int], object], b_blocks: Dict[Tuple[int, int], object], m: int, k: int,
                   n: int) -> Dict[Tuple[int, int], np.ndarray]:
    """BlockMatrix.multiply(other: BlockMatrix) on equal inner grids (BlockMatrix.scala:152-186) with sparse blocks:
    every product (i, j, kk) through block_product, the k partials of a C block summed in kk order (reduceByKey add,
    one rounding per partial)."""
    out = {}
    for i in range(m):
        for j in range(n):
            acc = None
            for kk in range(k):
                p = block_product(a_blocks[(i, kk)], b_blocks[(kk, j)])
                acc = p if acc is None else acc + p
            out[(i, j)] = acc
    return out
