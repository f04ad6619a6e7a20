"""SparseMatrix and LibMatrixMult — matrix/Matrices.scala:136-253 and matrix/LibMatrixMult.scala, device resident.

The reference keeps a sparse block as one SparseVector per column; here the same matrix is CSC in HBM (an `mb_spblock` of
the C ABI: col_ptr, row_idx, val).  Every product writes a dense block, as the reference does, and is bit-identical to the
reference's loop: each output element is a sequential sum from +0.0 in the reference's term order, one rounded multiply
and one rounded add per term.  The one documented deviation is LibMatrixMult.multSparseDense, which is computed as
defined (Breeze's `*`) rather than with the reference's out-of-range indexing (DESIGN.md, documented deviations).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np

from .. import _native as nat
from ..runtime import Runtime


def _i32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.int32))


class SparseMatrix:
    """A (numRows x numCols) CSC block on the GPU.  `values` is the reference's constructor argument: one entry per column,
    each None (an empty column) or an (indices, values) pair like a SparseVector."""

    def __init__(self, numRows: int, numCols: int, values: Optional[Sequence] = None, *, _handle=None):
        self._rows, self._cols = int(numRows), int(numCols)
        self._handle = None
        if _handle is not None:
            self._handle = _handle
            return
        col_ptr = np.zeros(self._cols + 1, dtype=np.int64)
        idx, val = [], []
        for c, sv in enumerate(values if values is not None else [None] * self._cols):
            if sv is not None:
                i, v = sv
                idx.append(np.asarray(i, dtype=np.int64).reshape(-1))
                val.append(np.asarray(v, dtype=np.float64).reshape(-1))
                if idx[-1].shape != val[-1].shape:
                    raise nat.MarlinArgumentError(nat.MB_ERR_INVALID_ARG, f"column {c}: {idx[-1].size} indices, "
                                                  f"{val[-1].size} values")
                col_ptr[c + 1] = idx[-1].size
        if values is not None and len(values) != self._cols:
            raise nat.MarlinArgumentError(nat.MB_ERR_INVALID_ARG, f"{len(values)} column vectors for {self._cols} columns")
        col_ptr = np.cumsum(col_ptr)
        row_idx = np.concatenate(idx) if idx else np.zeros(0, dtype=np.int64)
        data = np.concatenate(val) if val else np.zeros(0)
        self._upload(col_ptr, row_idx, data)

    @classmethod
    def fromCSC(cls, numRows: int, numCols: int, colPtr, rowIndices, data) -> "SparseMatrix":
        out = cls.__new__(cls)
        out._rows, out._cols, out._handle = int(numRows), int(numCols), None
        out._upload(np.asarray(colPtr), np.asarray(rowIndices), np.asarray(data))
        return out

    @classmethod
    def fromScipy(cls, m) -> "SparseMatrix":
        """From a scipy.sparse matrix (converted to CSC with sorted indices)."""
        csc = m.tocsc()
        csc.sort_indices()
        return cls.fromCSC(csc.shape[0], csc.shape[1], csc.indptr, csc.indices, csc.data)

    def _upload(self, col_ptr, row_idx, data) -> None:
        if col_ptr.size != self._cols + 1 or (col_ptr.size and col_ptr[-1] >= 2 ** 31):
            raise nat.MarlinArgumentError(nat.MB_ERR_INVALID_ARG, "sparse block: col_ptr needs numCols + 1 entries below 2^31")
        if row_idx.size != data.size or row_idx.size != int(col_ptr[-1]):
            raise nat.MarlinArgumentError(nat.MB_ERR_INVALID_ARG, "sparse block: row_idx / values do not match col_ptr")
        if row_idx.size and (row_idx.min() < -2 ** 31 or row_idx.max() >= 2 ** 31):
            raise nat.MarlinArgumentError(nat.MB_ERR_INVALID_ARG, "sparse block: row index outside int32")
        cp, ri, v = _i32(col_ptr), _i32(row_idx), np.ascontiguousarray(data, dtype=np.float64)
        rt = Runtime.get(); rt.sync_stream()
        h = nat.c_sp()
        nat.check(rt.lib.mb_spblock_upload(rt.ctx, self._rows, self._cols, cp.ctypes.data_as(C.POINTER(C.c_int32)),
                                           ri.ctypes.data_as(C.POINTER(C.c_int32)), v.ctypes.data_as(nat.c_dp), C.byref(h)))
        self._handle = h

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None:
            try:
                rt = Runtime._instance
                if rt is not None:
                    rt.lib.mb_spblock_free(rt.ctx, h)
            except Exception:
                pass

    # ---- reference accessors
    @property
    def numRows(self) -> int:
        return self._rows

    @property
    def numCols(self) -> int:
        return self._cols

    @property
    def nnz(self) -> int:
        n = C.c_int64()
        nat.check(nat.load().mb_spblock_info(self._handle, None, None, C.byref(n)))
        return int(n.value)

    def handle(self):
        return self._handle

    def csc(self) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """Download (col_ptr, row_idx, values)."""
        nnz = self.nnz
        cp = np.zeros(self._cols + 1, dtype=np.int32)
        ri = np.zeros(max(nnz, 1), dtype=np.int32)
        v = np.zeros(max(nnz, 1), dtype=np.float64)
        rt = Runtime.get(); rt.sync_stream()
        nat.check(rt.lib.mb_spblock_download(rt.ctx, self._handle, cp.ctypes.data_as(C.POINTER(C.c_int32)),
                                             ri.ctypes.data_as(C.POINTER(C.c_int32)), v.ctypes.data_as(nat.c_dp)))
        return cp, ri[:nnz], v[:nnz]

    def toBreeze(self):
        """Matrices.scala:149-183 (Breeze CSCMatrix) -> scipy.sparse.csc_matrix on the host."""
        import scipy.sparse as sps
        cp, ri, v = self.csc()
        return sps.csc_matrix((v, ri, cp), shape=(self._rows, self._cols))

    def toDense(self, out=None):
        """Matrices.scala:185-198: the dense block (a SubMatrix on the GPU)."""
        from .sub_matrix import SubMatrix
        rt = Runtime.get(); rt.sync_stream()
        if out is None:
            out = SubMatrix.empty(self._rows, self._cols, nat.MB_F64)
        nat.check(rt.lib.mb_spblock_to_dense(rt.ctx, self._handle, out.handle()))
        return out

    def multiply(self, other: "SparseMatrix", out=None, accumulate: bool = False):
        """Matrices.scala:208-231: sparse x sparse -> dense block."""
        from .sub_matrix import SubMatrix
        rt = Runtime.get(); rt.sync_stream()
        if out is None:
            out = SubMatrix.empty(self._rows, other._cols, nat.MB_F64)
        nat.check(rt.lib.mb_spgemm_to_dense(rt.ctx, self._handle, other._handle, out.handle(), int(accumulate)))
        return out

    def _map_values(self, alpha: float, beta: float, divide_by: Optional[float] = None) -> "SparseMatrix":
        """The scalar ops of SubMatrix.scala:52-58,71-85,121-129: a copy whose STORED values are alpha*v + beta (or v / b)."""
        rt = Runtime.get(); rt.sync_stream()
        h = nat.c_sp()
        nat.check(rt.lib.mb_spblock_copy(rt.ctx, self._handle, C.byref(h)))
        out = SparseMatrix(self._rows, self._cols, _handle=h)
        if self.nnz:
            src, dst = nat.c_blk(), nat.c_blk()
            nat.check(rt.lib.mb_spblock_values(rt.ctx, self._handle, C.byref(src)))
            nat.check(rt.lib.mb_spblock_values(rt.ctx, out._handle, C.byref(dst)))
            try:
                if divide_by is not None:
                    nat.check(rt.lib.mb_block_div(rt.ctx, src, float(divide_by), 0, dst))
                else:
                    nat.check(rt.lib.mb_block_axpb(rt.ctx, src, float(alpha), float(beta), dst))
            finally:
                rt.lib.mb_block_free(rt.ctx, src)
                rt.lib.mb_block_free(rt.ctx, dst)
        return out

    @staticmethod
    def randCount(numRows: int, numCols: int, sparsity: float) -> int:
        """Entries per column of rand(numRows, numCols, sparsity): (numCols * sparsity).toInt, checked."""
        n = C.c_int32()
        nat.check(nat.load().mb_sparse_rand_count(int(numRows), int(numCols), float(sparsity), C.byref(n)))
        return int(n.value)

    @staticmethod
    def rand(numRows: int, numCols: int, sparsity: float, seed: Optional[int] = None) -> "SparseMatrix":
        """Matrices.scala:236-253, generated on the GPU.  The reference is unseeded; `seed` (a partition seed, as from
        MTUtils' per-block seeds) makes the matrix reproducible: column c has its own splitmix64 stream, rows are drawn by
        selection sampling (sorted, distinct, exactly (numCols*sparsity).toInt per column), values U[0,1)."""
        if seed is None:
            import time
            seed = time.time_ns()
        rt = Runtime.get(); rt.sync_stream()
        h = nat.c_sp()
        nat.check(rt.lib.mb_spblock_rand(rt.ctx, int(numRows), int(numCols), float(sparsity), int(seed), C.byref(h)))
        return SparseMatrix(numRows, numCols, _handle=h)

    def __repr__(self):
        return f"SparseMatrix({self._rows}x{self._cols}, nnz={self.nnz})"


class LibMatrixMult:
    """matrix/LibMatrixMult.scala"""

    @staticmethod
    def multDenseSparse(denseMat, sparseMat: SparseMatrix, out=None, accumulate: bool = False):
        """:15-41 — dense x sparse -> dense block, the single-1.0-column copy shortcut (:28-29) included."""
        from .sub_matrix import SubMatrix
        a = denseMat if isinstance(denseMat, SubMatrix) else SubMatrix(denseMat)
        rt = Runtime.get(); rt.sync_stream()
        if out is None:
            if accumulate:
                raise ValueError("accumulate needs an output block")
            out = SubMatrix.empty(a.rows, sparseMat.numCols, nat.MB_F64)
        nat.check(rt.lib.mb_spmm_dense_sparse(rt.ctx, a.handle(), sparseMat.handle(), out.handle(), int(accumulate)))
        return out

    @staticmethod
    def multSparseDense(sparseMat: SparseMatrix, denseMat, out=None, accumulate: bool = False):
        """:43-77 as defined: C(r,j) = sum over k ascending of A(r,k)*B(k,j) (the reference indexes B out of range once
        K or N exceeds 32; see DESIGN.md).  Views (slices, transposes) of B are read as views."""
        from .sub_matrix import SubMatrix
        b = denseMat if isinstance(denseMat, SubMatrix) else SubMatrix(denseMat)
        rt = Runtime.get(); rt.sync_stream()
        if out is None:
            if accumulate:
                raise ValueError("accumulate needs an output block")
            out = SubMatrix.empty(sparseMat.numRows, b.cols, nat.MB_F64)
        nat.check(rt.lib.mb_spmm_sparse_dense(rt.ctx, sparseMat.handle(), b.handle(), out.handle(), int(accumulate)))
        return out
