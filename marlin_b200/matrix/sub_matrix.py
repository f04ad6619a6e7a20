"""SubMatrix — the per-block value type (matrix/SubMatrix.scala), device resident.

The reference's SubMatrix wraps a Breeze DenseMatrix[Double] on the JVM heap; here the same
(data, offset, rows, cols, majorStride, isTranspose) record points into HBM.  The buffer is a torch
tensor only so that torch.distributed (NCCL) can move it; every arithmetic method calls the C ABI
of libmarlin_b200.so (the kernel seam named in SURVEY.md §2 #3).  A sparse block (`SubMatrix(spMatrix=...)`) holds a
device-resident CSC SparseMatrix instead and dispatches exactly as SubMatrix.scala:41-139 does.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Union

import numpy as np
import torch

from .. import _native as nat
from ..runtime import Runtime

_TORCH_DTYPE = {nat.MB_F64: torch.float64, nat.MB_BF16: torch.bfloat16, nat.MB_F32: torch.float32}
_MB_DTYPE = {v: k for k, v in _TORCH_DTYPE.items()}

Number = Union[int, float]


def _unsupported(msg: str) -> nat.MarlinArgumentError:
    return nat.MarlinArgumentError(nat.MB_ERR_UNSUPPORTED, msg)


class SubMatrix:
    """A dense block.  Element (r, c) = buf.flatten()[offset + r + c*ld] (or [offset + c + r*ld] if
    is_transpose), exactly Breeze's DenseMatrix indexing.  Or, built with `spMatrix=`, a sparse block (CSC on the GPU)."""

    def __init__(self, denseMatrix=None, *, spMatrix=None, buf: Optional[torch.Tensor] = None, rows: int = 0, cols: int = 0,
                 ld: Optional[int] = None, offset: int = 0, is_transpose: bool = False, device=None):
        self._handle = None
        self._sp = spMatrix
        if spMatrix is not None:                                            # SubMatrix.scala:22-25
            self.buf = None
            self._rows, self._cols = spMatrix.numRows, spMatrix.numCols
            self.ld, self.offset, self.is_transpose = max(1, self._rows), 0, False
            return
        if denseMatrix is not None:
            if isinstance(denseMatrix, SubMatrix):
                src = denseMatrix
                buf, rows, cols, ld, offset, is_transpose = src.buf, src._rows, src._cols, src.ld, src.offset, src.is_transpose
            else:
                arr = np.asarray(denseMatrix, dtype=np.float64)
                if arr.ndim != 2:
                    raise ValueError("SubMatrix needs a 2-D dense matrix")
                rows, cols = arr.shape
                flat = np.ascontiguousarray(arr.T).reshape(-1)            # column-major data array
                t = torch.from_numpy(flat)
                if device is None:
                    device = Runtime.get().device if Runtime.available() else torch.device("cpu")
                buf = t.to(device)
                ld, offset, is_transpose = max(1, rows), 0, False
        if buf is None:
            raise ValueError("SubMatrix: no data")
        if not buf.is_contiguous():
            raise ValueError("SubMatrix buffer must be contiguous")
        self.buf = buf
        self._rows, self._cols = int(rows), int(cols)
        self.ld = int(ld if ld is not None else max(1, (cols if is_transpose else rows)))
        self.offset = int(offset)
        self.is_transpose = bool(is_transpose)

    # ---- construction helpers ----
    @staticmethod
    def empty(rows: int, cols: int, dtype: int = nat.MB_F64, device=None) -> "SubMatrix":
        if device is None:
            device = Runtime.get().device
        buf = torch.empty(max(1, rows) * max(0, cols) if rows * cols else 0, dtype=_TORCH_DTYPE[dtype], device=device)
        return SubMatrix(buf=buf, rows=rows, cols=cols, ld=max(1, rows))

    @staticmethod
    def zeros(rows: int, cols: int, dtype: int = nat.MB_F64, device=None) -> "SubMatrix":
        out = SubMatrix.empty(rows, cols, dtype, device)
        out.buf.zero_()
        return out

    # ---- reference accessors (matrix/SubMatrix.scala:27-39) ----
    @property
    def rows(self) -> int:
        return self._rows

    @property
    def cols(self) -> int:
        return self._cols

    @property
    def isSparse(self) -> bool:
        return self._sp is not None

    @property
    def denseBlock(self) -> Optional["SubMatrix"]:
        return None if self._sp is not None else self

    @property
    def sparseBlock(self):
        return self._sp

    @property
    def dtype(self) -> int:
        return nat.MB_F64 if self._sp is not None else _MB_DTYPE[self.buf.dtype]

    @property
    def t(self) -> "SubMatrix":
        """Breeze `.t`: a transposed view, no copy."""
        if self._sp is not None:
            self.handle()                                                    # raises MB_ERR_UNSUPPORTED
        return SubMatrix(buf=self.buf, rows=self._cols, cols=self._rows, ld=self.ld, offset=self.offset,
                         is_transpose=not self.is_transpose)

    def slice(self, r0: int, r1: int, c0: int, c1: int) -> "SubMatrix":
        """Breeze `m(r0 until r1, c0 until c1)`: a view with the parent's majorStride (BlockMatrix.scala:198,299)."""
        if self._sp is not None:
            self.handle()                                                    # raises MB_ERR_UNSUPPORTED
        if not (0 <= r0 <= r1 <= self._rows and 0 <= c0 <= c1 <= self._cols):
            raise ValueError("slice out of range")
        rs, cs = (self.ld, 1) if self.is_transpose else (1, self.ld)
        return SubMatrix(buf=self.buf, rows=r1 - r0, cols=c1 - c0, ld=self.ld, offset=self.offset + r0 * rs + c0 * cs,
                         is_transpose=self.is_transpose)

    def is_packed(self) -> bool:
        return (not self.is_transpose) and self.offset == 0 and self.ld == max(1, self._rows)

    # ---- native handle ----
    def _dense_runtime(self) -> Runtime:
        """The runtime, synchronised to the current stream, for an operation on a dense block."""
        if self._sp is not None:
            self.handle()                                                    # raises MB_ERR_UNSUPPORTED
        rt = Runtime.get(); rt.sync_stream()
        return rt

    def handle(self):
        if self._sp is not None:
            raise _unsupported("this operation needs a dense block and this block is sparse: convert with toDenseBlocks")
        if self._handle is None:
            if not self.buf.is_cuda:
                raise nat.MarlinError(nat.MB_ERR_CUDA, "block lives in host memory: marlin_b200 computes on B200 only "
                                      "(no CPU fallback)")
            rt = Runtime.get()
            h = nat.c_blk()
            nat.check(rt.lib.mb_block_wrap(rt.ctx, C.c_void_p(self.buf.data_ptr()), self.offset, self._rows, self._cols,
                                           self.ld, int(self.is_transpose), self.dtype, C.byref(h)))
            self._handle = h
            ev = getattr(self, "_ready_event", None)
            if ev is not None:
                nat.check(rt.lib.mb_block_set_ready_event(h, C.c_void_p(ev.cuda_event)))
        return self._handle

    def mark_ready(self) -> "SubMatrix":
        """Record that everything queued so far on the current stream produces this block's FINAL contents (blocks are
        immutable values, like the blocks of a cached RDD): the multi-GPU multiply then offers the block to other ranks as
        soon as this event completes instead of after all later work on the stream (see mb_block_set_ready_event)."""
        if self._sp is None and self.buf.is_cuda:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.buf.device))
            self._ready_event = ev
            if self._handle is not None:
                rt = Runtime.get()
                nat.check(rt.lib.mb_block_set_ready_event(self._handle, C.c_void_p(ev.cuda_event)))
        return self

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None:
            try:
                rt = Runtime._instance
                if rt is not None:
                    rt.lib.mb_block_free(rt.ctx, h)
            except Exception:
                pass

    def _new_like(self, rows: Optional[int] = None, cols: Optional[int] = None, dtype: Optional[int] = None) -> "SubMatrix":
        """Result block for an element-wise op: same shape and the same storage orientation as `self`
        (a row-major DenseVecMatrix shard stays row-major, so the kernels take the flat 128-bit path)."""
        rows = self._rows if rows is None else rows
        cols = self._cols if cols is None else cols
        dtype = self.dtype if dtype is None else dtype
        if self.is_transpose:
            buf = torch.empty(rows * cols, dtype=_TORCH_DTYPE[dtype], device=self.buf.device)
            return SubMatrix(buf=buf, rows=rows, cols=cols, ld=max(1, cols), is_transpose=True)
        return SubMatrix.empty(rows, cols, dtype, self.buf.device)

    # ---- arithmetic (matrix/SubMatrix.scala:41-139) ----
    def _check_dense_pair(self, other: "SubMatrix", op: str) -> None:
        if self.isSparse or other.isSparse:                                  # :46-48, :66-68
            raise _unsupported(f"Not supported {op}-operator between matrices of sparsity with {str(self.isSparse).lower()} "
                               f"and {str(other.isSparse).lower()}")

    def add(self, other: Union["SubMatrix", Number]) -> "SubMatrix":
        if isinstance(other, SubMatrix):
            self._check_dense_pair(other, "add")
        elif self.isSparse:
            return SubMatrix(spMatrix=self._sp._map_values(1.0, float(other)))                   # :53-56
        rt = self._dense_runtime()
        out = self._new_like()
        if isinstance(other, SubMatrix):
            nat.check(rt.lib.mb_block_add(rt.ctx, self.handle(), other.handle(), out.handle()))      # :41-45
        else:
            nat.check(rt.lib.mb_block_axpb(rt.ctx, self.handle(), 1.0, float(other), out.handle()))   # :52-58
        return out

    def subtract(self, other: Union["SubMatrix", Number]) -> "SubMatrix":
        if isinstance(other, SubMatrix):
            self._check_dense_pair(other, "subtract")
        elif self.isSparse:
            return SubMatrix(spMatrix=self._sp._map_values(1.0, -float(other)))                  # :72-75
        rt = self._dense_runtime()
        out = self._new_like()
        if isinstance(other, SubMatrix):
            nat.check(rt.lib.mb_block_sub(rt.ctx, self.handle(), other.handle(), out.handle()))      # :60-64
        else:
            nat.check(rt.lib.mb_block_axpb(rt.ctx, self.handle(), 1.0, -float(other), out.handle()))  # :71-77
        return out

    def divide(self, b: Number) -> "SubMatrix":
        if self.isSparse:
            return SubMatrix(spMatrix=self._sp._map_values(1.0, 0.0, divide_by=float(b)))       # :80-83
        rt = self._dense_runtime()
        out = self._new_like()
        nat.check(rt.lib.mb_block_div(rt.ctx, self.handle(), float(b), 0, out.handle()))               # :79-85
        return out

    def subtractBy(self, b: Number) -> "SubMatrix":
        """b - x (matrix/BlockMatrix.scala:414-424; returns a new block instead of mutating in place)."""
        rt = self._dense_runtime()
        out = self._new_like()
        nat.check(rt.lib.mb_block_axpb(rt.ctx, self.handle(), -1.0, float(b), out.handle()))
        return out

    def divideBy(self, b: Number) -> "SubMatrix":
        """b / x (matrix/BlockMatrix.scala:442-452)."""
        rt = self._dense_runtime()
        out = self._new_like()
        nat.check(rt.lib.mb_block_div(rt.ctx, self.handle(), float(b), 1, out.handle()))
        return out

    def elementMultiply(self, other: "SubMatrix") -> "SubMatrix":
        rt = self._dense_runtime()
        out = self._new_like()
        nat.check(rt.lib.mb_block_hadamard(rt.ctx, self.handle(), other.handle(), out.handle()))
        return out

    def multiply(self, other, out: Optional["SubMatrix"] = None, accumulate: bool = False,
                 out_dtype: Optional[int] = None) -> "SubMatrix":
        """:87-111 (block x block, block x local matrix) and :123-131 (scalar).  With a sparse operand the four arms of
        :88-100 (dense x dense, sparse x sparse, dense x sparse, sparse x dense) and :112-114 (sparse x local matrix)."""
        if isinstance(other, (int, float)) and self.isSparse:
            return SubMatrix(spMatrix=self._sp._map_values(float(other), 0.0))                  # :122-125
        if not isinstance(other, (int, float)) and (self.isSparse or (isinstance(other, SubMatrix) and other.isSparse)):
            return self._multiply_sparse(other, out, accumulate)
        rt = self._dense_runtime()
        if isinstance(other, (int, float)):
            res = self._new_like()
            nat.check(rt.lib.mb_block_axpb(rt.ctx, self.handle(), float(other), 0.0, res.handle()))
            return res
        if not isinstance(other, SubMatrix):
            other = SubMatrix(other, device=self.buf.device)
        if out is None:
            if accumulate:
                raise ValueError("accumulate needs an output block")
            dt = out_dtype if out_dtype is not None else (nat.MB_F32 if self.dtype == nat.MB_BF16 else self.dtype)
            out = SubMatrix.empty(self._rows, other._cols, dt, self.buf.device)
        nat.check(rt.lib.mb_block_gemm(rt.ctx, self.handle(), other.handle(), out.handle(), int(accumulate)))
        return out

    def _multiply_sparse(self, other, out: Optional["SubMatrix"], accumulate: bool) -> "SubMatrix":
        from .sparse_matrix import LibMatrixMult
        if not isinstance(other, SubMatrix):
            other = SubMatrix(other)
        if self.isSparse and other.isSparse:
            return self._sp.multiply(other._sp, out=out, accumulate=accumulate)            # :92-94
        if other.isSparse:
            return LibMatrixMult.multDenseSparse(self, other._sp, out=out, accumulate=accumulate)   # :95-97
        return LibMatrixMult.multSparseDense(self._sp, other, out=out, accumulate=accumulate)      # :98-100, :112-114

    def toDenseBlock(self) -> "SubMatrix":
        """`new SubMatrix(denseMatrix = sparseBlock.toDense)` (BlockMatrix.scala:598); a dense block is returned as is."""
        return self._sp.toDense() if self._sp is not None else self

    def dot(self, other: "SubMatrix") -> float:
        """Breeze `v.t * w` of two single-column (or single-row) blocks (matrix/DistributedVector.scala:167)."""
        rt = self._dense_runtime()
        out = C.c_double()
        nat.check(rt.lib.mb_block_dot(rt.ctx, self.handle(), other.handle(), C.byref(out)))
        return float(out.value)

    def outer(self, other: "SubMatrix") -> "SubMatrix":
        """Breeze `v * w.t` (matrix/DistributedVector.scala:157): rank-1 block of two vectors."""
        rt = self._dense_runtime()
        n0 = self._rows * self._cols
        n1 = other._rows * other._cols
        out = SubMatrix.empty(n0, n1, nat.MB_F64, self.buf.device)
        nat.check(rt.lib.mb_block_ger(rt.ctx, self.handle(), other.handle(), out.handle()))
        return out

    # ---- factorizations: the Breeze/LAPACK calls of DenseVecMatrix.luDecompose / choleskyDecompose / inverse ----
    def lu(self):
        """`brzLU(m)` (matrix/DenseVecMatrix.scala:302): (packed unit-lower L and U, permutation array with the
        reference's meaning: row i of L*U is row perm[i] of this block)."""
        rt = self._dense_runtime()
        out = self.copy()
        perm = (C.c_int32 * max(1, self._rows))()
        nat.check(rt.lib.mb_block_lu(rt.ctx, out.handle(), perm))
        return out, np.array(perm[: self._rows], dtype=np.int64)

    def cholesky(self) -> "SubMatrix":
        """`brzCholesky(m)` (:495,513): lower L with L L^T = this, zeros above the diagonal."""
        rt = self._dense_runtime()
        out = self.copy()
        nat.check(rt.lib.mb_block_cholesky(rt.ctx, out.handle()))
        return out

    def inverse(self) -> "SubMatrix":
        """`brzInv(m)` (:587,606)."""
        rt = self._dense_runtime()
        out = SubMatrix.empty(self._rows, self._cols, nat.MB_F64, self.buf.device)
        nat.check(rt.lib.mb_block_inverse(rt.ctx, self.handle(), out.handle()))
        return out

    def solveTriangular(self, rhs: "SubMatrix", lower: bool, unit: bool = False) -> "SubMatrix":
        """`this \\ rhs` for a triangular `this` (the `l \\ ...` of :364): returns X with this * X = rhs."""
        rt = self._dense_runtime()
        x = rhs.copy()
        nat.check(rt.lib.mb_block_trsm(rt.ctx, self.handle(), int(lower), int(unit), x.handle()))
        return x

    def add_(self, other: "SubMatrix") -> "SubMatrix":
        """In-place accumulate (the reduceByKey combine of BlockMatrix.scala:177 without a new allocation)."""
        rt = self._dense_runtime()
        nat.check(rt.lib.mb_block_add(rt.ctx, self.handle(), other.handle(), self.handle()))
        return self

    def transpose(self) -> "SubMatrix":
        """`denseBlock.t.copy` (matrix/BlockMatrix.scala:517): materialised transpose."""
        rt = self._dense_runtime()
        out = SubMatrix.empty(self._cols, self._rows, self.dtype, self.buf.device)
        nat.check(rt.lib.mb_block_transpose(rt.ctx, self.handle(), out.handle()))
        return out

    def copy(self, dtype: Optional[int] = None) -> "SubMatrix":
        """Breeze `.copy`: packed column-major copy of a view (optionally converting fp64 <-> bf16/fp32)."""
        rt = self._dense_runtime()
        out = SubMatrix.empty(self._rows, self._cols, self.dtype if dtype is None else dtype, self.buf.device)
        nat.check(rt.lib.mb_block_copy(rt.ctx, self.handle(), out.handle()))
        return out

    def assign(self, src: "SubMatrix") -> None:
        """`this(range) := src` — copy src into this view."""
        rt = self._dense_runtime()
        nat.check(rt.lib.mb_block_copy(rt.ctx, src.handle(), self.handle()))

    def sum(self) -> float:
        rt = self._dense_runtime()
        blk = self if self.dtype == nat.MB_F64 else self.copy(nat.MB_F64)
        out = C.c_double()
        nat.check(rt.lib.mb_block_sum(rt.ctx, blk.handle(), C.byref(out)))
        return float(out.value)

    # ---- host transfer (toBreeze / collect) ----
    def toBreeze(self) -> np.ndarray:
        """Download as a (rows x cols) Fortran-ordered float64 ndarray (a sparse block is densified)."""
        if self._sp is not None:
            return self._sp.toDense().toBreeze()
        if self._rows == 0 or self._cols == 0:
            return np.zeros((self._rows, self._cols), order="F")
        if self.buf.is_cuda:
            blk = self if (self.is_packed() and self.dtype == nat.MB_F64) else self.copy(nat.MB_F64)
            flat = blk.buf[: self._rows * self._cols].cpu().numpy()
            return flat.reshape((self._rows, self._cols), order="F")
        # host-resident block (CPU-side plumbing tests only): pure indexing, no arithmetic
        flat = self.buf.to(torch.float64).numpy()
        r = np.arange(self._rows)[:, None]
        c = np.arange(self._cols)[None, :]
        idx = self.offset + (c + r * self.ld if self.is_transpose else r + c * self.ld)
        return np.asfortranarray(flat[idx])

    to_numpy = toBreeze

    def __repr__(self):
        if self._sp is not None:
            return f"SubMatrix(sparse {self._sp!r})"
        return f"SubMatrix({self._rows}x{self._cols}, ld={self.ld}, t={self.is_transpose}, {self.buf.dtype}, {self.buf.device})"


class RawBlock:
    """A column-major block at a raw device address that torch does not own — e.g. a staging slot in ANOTHER rank's HBM
    mapped through CUDA IPC.  Only usable as a GEMM output (`SubMatrix.multiply(..., out=RawBlock)`)."""

    def __init__(self, ptr: int, rows: int, cols: int, ld: int, dtype: int):
        self.ptr, self._rows, self._cols, self.ld, self._dtype = int(ptr), int(rows), int(cols), int(ld), int(dtype)
        self._handle = None

    @property
    def rows(self) -> int:
        return self._rows

    @property
    def cols(self) -> int:
        return self._cols

    @property
    def dtype(self) -> int:
        return self._dtype

    def slice(self, r0: int, r1: int, c0: int, c1: int) -> "RawBlock":
        esz = 8 if self._dtype == nat.MB_F64 else (4 if self._dtype == nat.MB_F32 else 2)
        return RawBlock(self.ptr + (r0 + c0 * self.ld) * esz, r1 - r0, c1 - c0, self.ld, self._dtype)

    def handle(self):
        if self._handle is None:
            rt = Runtime.get()
            h = nat.c_blk()
            nat.check(rt.lib.mb_block_wrap(rt.ctx, C.c_void_p(self.ptr), 0, self._rows, self._cols, self.ld, 0, self._dtype,
                                           C.byref(h)))
            self._handle = h
        return self._handle

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None:
            try:
                rt = Runtime._instance
                if rt is not None:
                    rt.lib.mb_block_free(rt.ctx, h)
            except Exception:
                pass
