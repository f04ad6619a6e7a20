"""BlockMatrix — the drop-in for edu.nju.pasalab.marlin.matrix.BlockMatrix (matrix/BlockMatrix.scala)
on the hot path: multiply / transpose / add and the conversions either side of them.

An RDD[(BlockID, SubMatrix)] becomes `blocks`: the (BlockID, SubMatrix) pairs THIS rank holds, plus a
`placement` callback (block -> rank) every rank agrees on.  With one process per GPU an RDD partition is a
GPU; Spark's shuffle for the multiply becomes grouped NCCL send/recv of tiles (marlin_b200.comm).
Method names, argument meaning and error behaviour follow the reference (Scala overloads are
dispatched on argument type).
"""
from __future__ import annotations

import math
from typing import Callable, Dict, Iterable, List, Optional, Tuple

import numpy as np
import torch

from .. import _native as nat
from .. import comm
from .. import peer
from .. import profiling
from ..runtime import Runtime, world
from .block import BlockID
from .distributed_matrix import DistributedMatrix
from .sub_matrix import SubMatrix


def _ceil_len(total: int, parts: int) -> int:
    return int(math.ceil(float(total) / float(parts)))


class BlockMatrix(DistributedMatrix):
    def __init__(self, blocks: Iterable[Tuple[BlockID, SubMatrix]], nRows: int = 0, nCols: int = 0, blksByRow: int = 0,
                 blksByCol: int = 0, placement: Optional[Callable[[int, int], int]] = None):
        self.blocks: List[Tuple[BlockID, SubMatrix]] = [(b if isinstance(b, BlockID) else BlockID(*b), s) for b, s in blocks]
        self._nRows, self._nCols, self._blksByRow, self._blksByCol = int(nRows), int(nCols), int(blksByRow), int(blksByCol)
        self._placement = placement

    # ------------------------------------------------------------------ dims (:36-67)
    def _all_gather_meta(self, items: list) -> list:
        """Metadata-only gather for lazily derived dims (the reference runs a Spark job here, :38,46,54,62)."""
        rank, ws = world()
        if ws == 1:
            return items
        import torch.distributed as dist
        out = [None] * ws
        dist.all_gather_object(out, items)
        return [x for part in out for x in part]

    def numRows(self) -> int:
        if self._nRows <= 0:
            vals = self._all_gather_meta([s.rows for b, s in self.blocks if b.column == 0])
            if not vals:
                raise nat.MarlinError(nat.MB_ERR_EMPTY, "empty collection")
            self._nRows = int(sum(vals))
        return self._nRows

    def numCols(self) -> int:
        if self._nCols <= 0:
            vals = self._all_gather_meta([s.cols for b, s in self.blocks if b.row == 0])
            if not vals:
                raise nat.MarlinError(nat.MB_ERR_EMPTY, "empty collection")
            self._nCols = int(sum(vals))
        return self._nCols

    def numBlksByRow(self) -> int:
        if self._blksByRow <= 0:
            self._blksByRow = len(self._all_gather_meta([1 for b, s in self.blocks if b.column == 0]))
        return self._blksByRow

    def numBlksByCol(self) -> int:
        if self._blksByCol <= 0:
            self._blksByCol = len(self._all_gather_meta([1 for b, s in self.blocks if b.row == 0]))
        return self._blksByCol

    @property
    def getBlocks(self):
        return self.blocks

    # ------------------------------------------------------------------ sparse blocks
    def _any_sparse(self) -> bool:
        """Whether any block of this matrix (on any rank) is sparse; agreed once per matrix (blocks are immutable)."""
        if getattr(self, "_sparse", None) is None:
            self._sparse = any(self._all_gather_meta([any(s.isSparse for _, s in self.blocks)]))
        return self._sparse

    def _require_dense(self, op: str, *others) -> None:
        """The reference dereferences `denseBlock` here, which is null for a sparse block."""
        for m in (self,) + others:
            if isinstance(m, BlockMatrix) and m._any_sparse():
                raise nat.MarlinArgumentError(nat.MB_ERR_UNSUPPORTED, f"{op} is not supported on a BlockMatrix with sparse "
                                              "blocks: convert it with toDenseBlocks first")

    def toDenseBlocks(self) -> "BlockMatrix":
        """:596-603 — every sparse block becomes `new SubMatrix(denseMatrix = sparseBlock.toDense)` on its GPU."""
        res = [(b, s.toDenseBlock()) for b, s in self.blocks]
        return BlockMatrix(res, self._nRows, self._nCols, self._blksByRow, self._blksByCol, self._placement)

    def owner(self, row: int, col: int) -> int:
        """Rank holding block (row, col): explicit placement or MatrixElemOpPartitioner order mod G."""
        rank, ws = world()
        if ws == 1:
            return 0
        if self._placement is not None:
            return self._placement(row, col)
        return comm.elem_owner(row, col, self.numBlksByCol(), ws)

    def elementsCount(self) -> int:
        """:477-479 (blocks.count())"""
        return len(self._all_gather_meta([1 for _ in self.blocks]))

    # ------------------------------------------------------------------ collect (:70-85)
    def toBreeze(self) -> np.ndarray:
        m, n = self.numRows(), self.numCols()
        rl, cl = _ceil_len(m, self.numBlksByRow()), _ceil_len(n, self.numBlksByCol())
        local = [((b.row, b.column), s.toBreeze()) for b, s in self.blocks]
        mat = np.zeros((m, n), order="F")
        for (r, c), arr in self._all_gather_meta(local):
            mat[r * rl:r * rl + arr.shape[0], c * cl:c * cl + arr.shape[1]] = arr
        return mat

    # ------------------------------------------------------------------ multiply overloads
    def multiply(self, other, *args, **kwargs):
        """Dispatch of the Scala overloads:
           multiply(other: BlockMatrix)                                   :149
           multiply(other: DistributedMatrix, cores: Int, thr: Int = 300) :87
           multiply(other: DistributedMatrix, splitMode: (Int,Int,Int))   :131
           multiply(b: Double)                                            :229
           multiply(B: BDM[Double])                                       :280
           multiply(v: DistributedVector) / multiply(v: BDV[Double])      :240 / :265"""
        from .dense_vec_matrix import DenseVecMatrix
        from .distributed_vector import DistributedVector
        if isinstance(other, (int, float)) and not args:
            return self._scalar("multiply", float(other))
        if isinstance(other, DistributedVector):
            return self._multiply_dist_vector(other)                      # multiply(v: DistributedVector) :240
        if isinstance(other, np.ndarray) and other.ndim == 1:
            return self._multiply_vector(other)                           # multiply(v: BDV[Double]) :265
        if isinstance(other, np.ndarray) or isinstance(other, SubMatrix):
            return self._multiply_local(other)
        if args and isinstance(args[0], (tuple, list)):
            return self._multiply_split(other, tuple(args[0]))
        if "splitMode" in kwargs:
            return self._multiply_split(other, tuple(kwargs["splitMode"]))
        if args or "cores" in kwargs:
            cores = args[0] if args else kwargs["cores"]
            thr = args[1] if len(args) > 1 else kwargs.get("broadcastThreshold", 300)
            return self._multiply_auto(other, int(cores), int(thr))
        if isinstance(other, BlockMatrix):
            return self._multiply_block(other)
        if isinstance(other, DenseVecMatrix):
            raise TypeError("multiply(DenseVecMatrix) needs `cores` or a splitMode, as in the reference API")
        raise TypeError(f"multiply: unsupported operand {type(other)}")

    def _multiply_auto(self, other, cores: int, broadcastThreshold: int = 300):
        """:87-122"""
        from .dense_vec_matrix import DenseVecMatrix
        if self.numCols() != other.numRows():
            raise nat.MarlinArgumentError(nat.MB_ERR_DIM_MISMATCH, "Dimension mismatch during matrix-matrix multiplication: "
                                          f"{self.numCols()} vs {other.numRows()}")
        import ctypes as C
        lib = nat.load()
        strat = C.c_int32()
        mkn = (C.c_int32 * 3)()
        nat.check(lib.mb_choose_strategy(self.numRows(), self.numCols(), other.numCols(), cores, broadcastThreshold,
                                         int(isinstance(other, BlockMatrix)), C.byref(strat), mkn))
        if strat.value == 0:
            return self._multiply_local(other.toBreeze())
        if strat.value == 1:
            if isinstance(other, DenseVecMatrix):
                # reference quirk (:97-98): evaluates that.multiply(this.toBreeze()), i.e. B * A_local
                return other.multiply(self.toBreeze())
            return other.multiplyBy(self.toBreeze())                             # :114-115
        return self._multiply_split(other, (mkn[0], mkn[1], mkn[2]))

    def _multiply_split(self, other, splitMode: Tuple[int, int, int]) -> "BlockMatrix":
        """:131-147"""
        if self.numCols() != other.numRows():
            raise nat.MarlinArgumentError(nat.MB_ERR_DIM_MISMATCH, "Dimension mismatch during matrix-matrix multiplication: "
                                          f"{self.numCols()} vs {other.numRows()}")
        m, k, n = splitMode
        return self.toBlockMatrix(m, k)._multiply_block(other.toBlockMatrix(k, n))

    def _multiply_block(self, other: "BlockMatrix") -> "BlockMatrix":
        """multiply(other: BlockMatrix) :149-220."""
        if self.numCols() != other.numRows():
            raise nat.MarlinArgumentError(nat.MB_ERR_DIM_MISMATCH, "Dimension mismatch during matrix-matrix multiplication: "
                                          f"{self.numCols()} vs {other.numRows()}")
        if self.numBlksByCol() == other.numBlksByRow():
            return self._multiply_same_grid(other)
        self._require_dense("multiply with a re-split grid (slices of denseBlock, :187-216)", other)
        if self.numBlksByCol() % other.numBlksByRow() == 0:                    # :187-201
            self._check_even_cols()
            ratio = self.numBlksByCol() // other.numBlksByRow()
            blks = []
            for b, mat in other.blocks:
                for i in range(ratio):
                    blks.append((BlockID(b.row * ratio + i, b.column),
                                 mat.slice(i * mat.rows // ratio, (i + 1) * mat.rows // ratio, 0, mat.cols)))
            split = BlockMatrix(blks, placement=lambda r, c, o=other, q=ratio: o.owner(r // q, c))
            return self._multiply_block(split)
        if other.numBlksByRow() % self.numBlksByCol() == 0:                    # :202-216 (row slices of `this`, as written)
            self._check_even_cols()
            ratio = other.numBlksByRow() // self.numBlksByCol()
            blks = []
            for b, mat in self.blocks:
                for i in range(ratio):
                    blks.append((BlockID(b.row * ratio + i, b.column),
                                 mat.slice(i * mat.rows // ratio, (i + 1) * mat.rows // ratio, 0, mat.cols)))
            split = BlockMatrix(blks, placement=lambda r, c, o=self, q=ratio: o.owner(r // q, c))
            return split._multiply_block(other)
        raise nat.MarlinArgumentError(nat.MB_ERR_UNSUPPORTED, "currently not supported for the two dimension of matrices")

    def _check_even_cols(self):
        if self.numCols() % self.numBlksByCol() != 0:
            raise nat.MarlinArgumentError(nat.MB_ERR_UNSUPPORTED, "only supported BlockMatrix which all the sub-matrices have the same cols")
        if (self.numCols() // self.numBlksByCol()) % 2 != 0:
            raise nat.MarlinArgumentError(nat.MB_ERR_UNSUPPORTED, "only supported sub-matrices with even number cols")

    def _multiply_same_grid(self, other: "BlockMatrix") -> "BlockMatrix":
        """:152-186 — m*k*n block products keyed by seq, k-way sum per C tile."""
        m, k, n = self.numBlksByRow(), self.numBlksByCol(), other.numBlksByCol()
        rank, ws = world()
        sparse = self._any_sparse() or other._any_sparse()
        if sparse and ws > 1:
            raise nat.MarlinArgumentError(nat.MB_ERR_UNSUPPORTED, "multiply of a BlockMatrix with sparse blocks runs on one "
                                          "rank; convert with toDenseBlocks for the multi-GPU multiply")
        plan = comm.plan_multiply(m, k, n, ws, self.owner, other.owner)
        a_local = {(b.row, b.column): s for b, s in self.blocks}
        b_local = {(b.row, b.column): s for b, s in other.blocks}
        a_tiles: Dict[Tuple[int, int], SubMatrix] = dict(a_local)
        b_tiles: Dict[Tuple[int, int], SubMatrix] = dict(b_local)
        M, N = self.numRows(), other.numCols()
        if ws > 1 and Runtime.available():
            mesh = peer.PeerMesh.get()
            if mesh is not None:
                res = self._multiply_p2p(other, mesh, plan, a_local, b_local)
                if res is not None:
                    return res
        if ws > 1:
            # tile replication (the two partitionBy shuffles of :165,171) as one grouped NCCL batch
            K = self.numCols()
            bm, bk, bn = _ceil_len(M, m), _ceil_len(K, k), _ceil_len(N, n)
            dims_a = lambda i, kk: (min(bm, M - i * bm), min(bk, K - kk * bk))
            dims_b = lambda kk, j: (min(bk, K - kk * bk), min(bn, N - j * bn))
            sends = [(s, d, ("A",) + key) for s, d, key in plan.a_sends] + [(s, d, ("B",) + key) for s, d, key in plan.b_sends]
            send_bufs, keep = {}, []
            for s, d, key in sends:
                if s == rank and key not in send_bufs:
                    src = (a_local if key[0] == "A" else b_local)[key[1:]]
                    if not src.is_packed():
                        src = src.copy(); keep.append(src)
                    send_bufs[key] = src.buf[: src.rows * src.cols]
            dtype_a = self._global_dtype()
            dev = Runtime.get().device if Runtime.available() else torch.device("cpu")

            def alloc(key):
                r, c = dims_a(*key[1:]) if key[0] == "A" else dims_b(*key[1:])
                return torch.empty(r * c, dtype=dtype_a, device=dev)

            with profiling.phase("exchange"):
                got = comm.exchange(sends, send_bufs, alloc, rank)
            for key, buf in got.items():
                r, c = dims_a(*key[1:]) if key[0] == "A" else dims_b(*key[1:])
                (a_tiles if key[0] == "A" else b_tiles)[key[1:]] = SubMatrix(buf=buf, rows=r, cols=c, ld=max(1, r))
        # the join + one dgemm per partition (:173-176), kk-partials of a C tile accumulated in place (:177)
        partial: Dict[Tuple[int, int], SubMatrix] = {}
        mine = plan.products.get(rank, [])
        by_c: Dict[Tuple[int, int], List[int]] = {}
        for (i, j, kk) in mine:
            by_c.setdefault((i, j), []).append(kk)
        # sparse operands: one sparse-product launch per block product, the kk partials accumulated in place
        whole = not sparse and bool(by_c) and all(sorted(v) == list(range(k)) for v in by_c.values())
        if whole and len(by_c) <= 16 and k <= 16:
            # this rank holds every kk of its C tiles: ONE grouped persistent launch (K loop concatenated over kk)
            import ctypes as C
            rt = Runtime.get(); rt.sync_stream()
            a_arr = (nat.c_blk * (m * k))()
            b_arr = (nat.c_blk * (k * n))()
            c_arr = (nat.c_blk * (m * n))()
            for (i, j) in by_c:
                for kk in range(k):
                    a_arr[i * k + kk] = a_tiles[(i, kk)].handle()
                    b_arr[kk * n + j] = b_tiles[(kk, j)].handle()
                a0, b0 = a_tiles[(i, 0)], b_tiles[(0, j)]
                out_dt = nat.MB_F32 if a0.dtype == nat.MB_BF16 else a0.dtype
                partial[(i, j)] = SubMatrix.empty(a0.rows, b0.cols, out_dt, a0.buf.device)
                c_arr[i * n + j] = partial[(i, j)].handle()
            ids = (C.c_int32 * len(by_c))(*[i * n + j for (i, j) in sorted(by_c)])
            with profiling.phase("gemm"):
                nat.check(rt.lib.mb_matmul_blocked_subset(rt.ctx, a_arr, b_arr, m, k, n, c_arr, ids, len(by_c)))
        else:
            for (i, j, kk) in mine:
                a, b = a_tiles[(i, kk)], b_tiles[(kk, j)]
                with profiling.phase("gemm"):
                    if (i, j) in partial:
                        a.multiply(b, out=partial[(i, j)], accumulate=True)
                    else:
                        partial[(i, j)] = a.multiply(b)
        if ws > 1 and plan.c_reduces:
            # reduceByKey across ranks (:177): partials travel to the C tile's owner and are added there
            sends = [(s, d, ("C",) + key + (s,)) for s, d, key in plan.c_reduces]
            send_bufs = {("C",) + key + (rank,): partial[key].buf[: partial[key].rows * partial[key].cols]
                         for s, d, key in plan.c_reduces if s == rank}

            def alloc_c(key):
                p = partial[key[1:3]]
                return torch.empty(p.rows * p.cols, dtype=p.buf.dtype, device=p.buf.device)

            with profiling.phase("reduce"):
                got = comm.exchange(sends, send_bufs, alloc_c, rank)
                for key, buf in sorted(got.items()):
                    p = partial[key[1:3]]
                    p.add_(SubMatrix(buf=buf, rows=p.rows, cols=p.cols, ld=max(1, p.rows)))
            for s, d, key in plan.c_reduces:
                if s == rank:
                    partial.pop(key, None)
        result = [(BlockID(i, j), blk) for (i, j), blk in sorted(partial.items())]
        owners = dict(plan.c_owner)
        return BlockMatrix(result, M, N, m, n, placement=(lambda r, c, o=owners: o[(r, c)]) if ws > 1 else None)

    # ------------------------------------------------------------------ NVLink peer-memory path
    def _multiply_p2p(self, other: "BlockMatrix", mesh, plan, a_local: dict, b_local: dict) -> Optional["BlockMatrix"]:
        """The multiply of :152-186 on the C-ABI engine (`mb_matmul_blocked_dist`, csrc/dist.cu): mapping of the m*k*n
        products to ranks, tile pulls over NVLink peer memory, the DMMA products and the reduce of the k partials all
        happen behind the ABI; this method only describes who owns what and allocates the C tiles this rank will own."""
        import ctypes as C
        rank = mesh.rank
        m, k, n = plan.m, plan.k, plan.n
        M, K, N = self.numRows(), self.numCols(), other.numCols()
        bm, bk, bn = _ceil_len(M, m), _ceil_len(K, k), _ceil_len(N, n)
        row_len = (C.c_int32 * m)(*[min(bm, M - i * bm) for i in range(m)])
        k_len = (C.c_int32 * k)(*[min(bk, K - kk * bk) for kk in range(k)])
        col_len = (C.c_int32 * n)(*[min(bn, N - j * bn) for j in range(n)])
        tdt = self._global_dtype()
        if tdt not in (torch.float64, torch.bfloat16):
            return None                                         # fp32 tiles: NCCL path (every rank takes the same branch)
        dt = nat.MB_F64 if tdt == torch.float64 else nat.MB_BF16
        out_dt = nat.MB_F64 if tdt == torch.float64 else nat.MB_F32
        rt = Runtime.get()
        rt.sync_stream()
        a_arr = (nat.c_blk * (m * k))()
        b_arr = (nat.c_blk * (k * n))()
        c_arr = (nat.c_blk * (m * n))()
        a_own = (C.c_int32 * (m * k))(*[self.owner(i, kk) for i in range(m) for kk in range(k)])
        b_own = (C.c_int32 * (k * n))(*[other.owner(kk, j) for kk in range(k) for j in range(n)])
        for (i, kk), s in a_local.items():
            a_arr[i * k + kk] = s.handle()
        for (kk, j), s in b_local.items():
            b_arr[kk * n + j] = s.handle()
        _, c_owner = mesh.plan(m, k, n)
        partial: Dict[Tuple[int, int], SubMatrix] = {}
        for i in range(m):
            for j in range(n):
                if c_owner[i * n + j] == rank:
                    partial[(i, j)] = SubMatrix.empty(row_len[i], col_len[j], out_dt, rt.device)
                    c_arr[i * n + j] = partial[(i, j)].handle()
        with profiling.phase("gemm"):
            nat.check(rt.lib.mb_matmul_blocked_dist(mesh.comm, a_arr, a_own, b_arr, b_own, m, k, n, row_len, k_len, col_len, dt, c_arr))
        result = [(BlockID(i, j), blk.mark_ready()) for (i, j), blk in sorted(partial.items())]
        owners = {(i, j): c_owner[i * n + j] for i in range(m) for j in range(n)}
        return BlockMatrix(result, M, N, m, n, placement=lambda r, c, o=owners: o[(r, c)])

    def inverse(self) -> "BlockMatrix":
        """inverse() :527-531 — toDenseVecMatrix().inverse()"""
        return self.toDenseVecMatrix().inverse()

    def _local_dtype(self):
        for _, s in self.blocks:
            return s.buf.dtype
        return torch.float64

    def _global_dtype(self):
        """Element type of the tiles, agreed by all ranks (a rank may hold no tile of this matrix)."""
        if getattr(self, "_gdtype", None) is None:
            names = self._all_gather_meta([str(s.buf.dtype) for _, s in self.blocks[:1]])
            self._gdtype = {"torch.float64": torch.float64, "torch.bfloat16": torch.bfloat16,
                            "torch.float32": torch.float32}[names[0]] if names else torch.float64
        return self._gdtype

    def _multiply_local(self, B) -> "BlockMatrix":
        """multiply(B: BDM[Double]) :280-303 — B is replicated on every rank (sc.broadcast)."""
        Bd = B if isinstance(B, SubMatrix) else None
        b_rows = Bd.rows if Bd is not None else B.shape[0]
        b_cols = Bd.cols if Bd is not None else B.shape[1]
        if self.numCols() != b_rows:
            raise nat.MarlinArgumentError(nat.MB_ERR_DIM_MISMATCH, "Dimension mismatch during matrix-matrix multiplication: "
                                          f"{self.numCols()} vs {b_rows}")
        if Bd is None:
            Bd = SubMatrix(B)
        if self.numBlksByCol() == 1:
            res = [(b, blk.multiply(Bd)) for b, blk in self.blocks]
            return BlockMatrix(res, self.numRows(), b_cols, self.numBlksByRow(), self.numBlksByCol(), self._placement)
        col_blk = _ceil_len(self.numCols(), self.numBlksByCol())
        acc: Dict[int, SubMatrix] = {}
        for b, blk in sorted(self.blocks, key=lambda t: (t[0].row, t[0].column)):
            start = b.column * col_blk
            end = self.numCols() if (b.column + 1) * col_blk > self.numCols() else (b.column + 1) * col_blk
            bs = Bd.slice(start, end, 0, b_cols)                       # Bb.value(startRow until endRow, ::) — a view
            if b.row in acc:
                blk.multiply(bs, out=acc[b.row], accumulate=True)
            else:
                acc[b.row] = blk.multiply(bs)
        rank, ws = world()
        if ws > 1:
            acc = self._reduce_row_partials(acc)
        res = [(BlockID(r, 0), blk) for r, blk in sorted(acc.items())]
        # the reference reports numBlksByCol() although every key has column 0 (:301); kept
        return BlockMatrix(res, self.numRows(), b_cols, self.numBlksByRow(), self.numBlksByCol(),
                           placement=(lambda r, c, s=self: s.owner(r, 0)) if ws > 1 else None)

    def _multiply_dist_vector(self, v):
        """multiply(v: DistributedVector) :240-259 — piece `id` of v meets every block of block column `id`
        (flatMap + join), block x piece on the GPU holding the block (mb_block_gemv), reduceByKey(add) over the block
        row: a running accumulate for the blocks one rank holds, then partials to the rank of block (row, 0).
        The result is labelled with v's length and split count, as the reference does (:252,257)."""
        from .distributed_vector import DistributedVector
        self._require_dense("matrix x vector multiply")            # SubMatrix.multiply(v: Vector), SubMatrix.scala:131-139
        if self.numCols() != v.length:
            raise nat.MarlinArgumentError(nat.MB_ERR_DIM_MISMATCH, "Dimension mismatch during matrix-matrix multiplication "
                                          f"{self.numCols()} v.s {v.length}")
        if self.numBlksByCol() != v.splitNum:
            raise nat.MarlinArgumentError(nat.MB_ERR_UNSUPPORTED, "not supported matrix or vector")
        pieces = v._replicated()
        acc: Dict[int, SubMatrix] = {}
        for b, blk in sorted(self.blocks, key=lambda t: (t[0].row, t[0].column)):
            x = pieces[b.column]
            if b.row in acc:
                blk.multiply(x, out=acc[b.row], accumulate=True)
            else:
                acc[b.row] = blk.multiply(x)
        rank, ws = world()
        if ws > 1 and self.numBlksByCol() != 1:
            acc = self._reduce_row_partials(acc)
        return DistributedVector(sorted(acc.items()), v.length, v.splitNum, placement=lambda i, s=self: s.owner(i, 0))

    def _multiply_vector(self, v: np.ndarray):
        """multiply(v: BDV[Double]) :265-274 — broadcast vector, the matrix must not be split by column."""
        from .distributed_vector import DistributedVector
        v = np.asarray(v, dtype=np.float64).reshape(-1)
        self._require_dense("matrix x vector multiply")            # SubMatrix.multiply(v: Vector), SubMatrix.scala:131-139
        if self.numCols() != v.shape[0]:
            raise nat.MarlinArgumentError(nat.MB_ERR_DIM_MISMATCH,
                                          f"matrix columns size {self.numCols()} not support vector length {v.shape[0]}")
        if self.numBlksByCol() != 1:
            raise nat.MarlinArgumentError(nat.MB_ERR_UNSUPPORTED, "should not split the matrix by column")
        x = SubMatrix(v.reshape(-1, 1))
        res = [(b.row, blk.multiply(x)) for b, blk in sorted(self.blocks, key=lambda t: t[0].row)]
        return DistributedVector(res, self.numRows(), self.numBlksByRow(), placement=lambda i, s=self: s.owner(i, 0))

    def multiplyBy(self, B) -> "BlockMatrix":
        """multiplyBy(B: BDM[Double]) :309-335 — a small local matrix times this block matrix (B replicated on every
        rank).  One block row: B * blk per block.  Several block rows: B(::, cols of block-row r) * blk, summed over r
        (reduceByKey on the unchanged BlockID, i.e. onto the block of row 0 ... as written, the keys keep their row, so
        only blocks with equal ids are summed — with distinct ids nothing is summed; reproduced as is).

        Two deliberate notes on labels: (1) for one block row the reference LABELS the result numRows() x B.cols (:319)
        although the blocks it holds are B.rows x numCols(); this port labels it with the dimensions of the data, B.rows x
        numCols() (what the several-block-rows branch at :333 also reports), so the result can be used by the next
        operation.  (2) The column range of B at :324-330 is bounded by numCols(), not by B.cols; when that range runs past
        B.cols Breeze's slice throws, and so does this port (no clamping)."""
        self._require_dense("multiplyBy")
        Bd = B if isinstance(B, SubMatrix) else SubMatrix(B)
        if Bd.cols != self.numRows():
            raise nat.MarlinArgumentError(nat.MB_ERR_DIM_MISMATCH, "Dimension mismatch during matrix-matrix multiplication: "
                                          f"{Bd.cols} vs {self.numRows()}")
        if self.numBlksByRow() == 1:
            res = [(b, Bd.multiply(blk)) for b, blk in self.blocks]                       # :315-319
            # the reference labels the result numRows() x B.cols (:319); the data is B.rows x numCols()
            return BlockMatrix(res, Bd.rows, self.numCols(), self.numBlksByRow(), self.numBlksByCol(), self._placement)
        row_blk = _ceil_len(self.numRows(), self.numBlksByRow())
        res = []
        for b, blk in self.blocks:
            start = b.row * row_blk
            end = self.numCols() if (b.row + 1) * row_blk > self.numCols() else (b.row + 1) * row_blk      # :324 bounds by numCols()
            if end > Bd.cols:                             # Breeze: B(::, start until end) out of bounds -> exception
                raise nat.MarlinArgumentError(nat.MB_ERR_INVALID_ARG, f"multiplyBy: column range {start} until {end} of the local "
                                              f"matrix is out of bounds ({Bd.cols} columns)")
            res.append((b, Bd.slice(0, Bd.rows, start, end).multiply(blk)))                               # :330-331
        return BlockMatrix(res, Bd.rows, self.numCols(), self.numBlksByRow(), self.numBlksByCol(), self._placement)

    def _reduce_row_partials(self, acc: Dict[int, SubMatrix]) -> Dict[int, SubMatrix]:
        """reduceByKey over column blocks held by different ranks (:300): partials go to owner(row, 0)."""
        rank, ws = world()
        k = self.numBlksByCol()
        sends = []
        for r in range(self.numBlksByRow()):
            dst = self.owner(r, 0)
            for src in sorted({self.owner(r, c) for c in range(k)}):
                if src != dst:
                    sends.append((src, dst, (r, src)))
        send_bufs = {(r, rank): acc[r].buf[: acc[r].rows * acc[r].cols] for s, d, (r, _) in sends if s == rank}
        bm = _ceil_len(self.numRows(), self.numBlksByRow())

        def alloc(key):
            r = key[0]
            if r in acc:
                p = acc[r]
                return torch.empty(p.rows * p.cols, dtype=p.buf.dtype, device=p.buf.device)
            raise RuntimeError("row partial owner holds no local partial")     # owner(r,0) always holds column 0

        got = comm.exchange(sends, send_bufs, alloc, rank)
        for (r, src), buf in sorted(got.items()):
            p = acc[r]
            p.add_(SubMatrix(buf=buf, rows=p.rows, cols=p.cols, ld=max(1, p.rows)))
        return {r: blk for r, blk in acc.items() if self.owner(r, 0) == rank}

    # ------------------------------------------------------------------ element-wise
    def _scalar(self, op: str, b: float) -> "BlockMatrix":
        if op in ("subtractBy", "divideBy"):
            self._require_dense(op)                                          # :416,444 read denseBlock.data
        f = {"add": lambda s: s.add(b), "subtract": lambda s: s.subtract(b), "multiply": lambda s: s.multiply(b),
             "divide": lambda s: s.divide(b), "subtractBy": lambda s: s.subtractBy(b), "divideBy": lambda s: s.divideBy(b)}[op]
        return BlockMatrix([(k, f(v)) for k, v in self.blocks], self.numRows(), self.numCols(), self.numBlksByRow(),
                           self.numBlksByCol(), self._placement)

    def _binary(self, other, op: str):
        from .dense_vec_matrix import DenseVecMatrix
        if isinstance(other, (int, float)):
            return self._scalar(op, float(other))
        if self.numRows() != other.numRows() or self.numCols() != other.numCols():
            raise nat.MarlinArgumentError(nat.MB_ERR_DIM_MISMATCH, "matrix dimension mismatch")
        self._require_dense(op, other)
        if isinstance(other, DenseVecMatrix):                                  # :346-349
            return getattr(self.toDenseVecMatrix(), op)(other)
        if self.numBlksByRow() != other.numBlksByRow() or self.numBlksByCol() != other.numBlksByCol():
            return getattr(self.toDenseVecMatrix(), op)(other.toDenseVecMatrix())          # :353-354
        rank, ws = world()
        theirs = {(b.row, b.column): s for b, s in other.blocks}
        if ws > 1:
            # blocks.join(mat.blocks): co-locate `other`'s blocks with ours (:356)
            sends = []
            for r in range(self.numBlksByRow()):
                for c in range(self.numBlksByCol()):
                    s, d = other.owner(r, c), self.owner(r, c)
                    if s != d:
                        sends.append((s, d, (r, c)))
            send_bufs = {}
            for s, d, key in sends:
                if s == rank:
                    blk = theirs[key] if theirs[key].is_packed() else theirs[key].copy()
                    send_bufs[key] = blk.buf[: blk.rows * blk.cols]
            mine = {(b.row, b.column): s for b, s in self.blocks}

            def alloc(key):
                p = mine[key]
                return torch.empty(p.rows * p.cols, dtype=p.buf.dtype, device=p.buf.device)

            for key, buf in comm.exchange(sends, send_bufs, alloc, rank).items():
                p = mine[key]
                theirs[key] = SubMatrix(buf=buf, rows=p.rows, cols=p.cols, ld=max(1, p.rows))
        fn = {"add": SubMatrix.add, "subtract": SubMatrix.subtract, "dotProduct": SubMatrix.elementMultiply}[op]
        res = [(b, fn(s, theirs[(b.row, b.column)])) for b, s in self.blocks if (b.row, b.column) in theirs]
        return BlockMatrix(res, self.numRows(), self.numCols(), self.numBlksByRow(), self.numBlksByCol(), self._placement)

    def add(self, other):
        """add(other: DistributedMatrix) :344-360, add(b: Double) :368-371"""
        return self._binary(other, "add")

    def subtract(self, other):
        """:380-407"""
        return self._binary(other, "subtract")

    def dotProduct(self, other):
        """:486-507 (element-wise product)"""
        return self._binary(other, "dotProduct")

    def divide(self, b: float) -> "BlockMatrix":
        """:432-435"""
        return self._scalar("divide", float(b))

    def subtractBy(self, b: float) -> "BlockMatrix":
        return self._scalar("subtractBy", float(b))

    def divideBy(self, b: float) -> "BlockMatrix":
        return self._scalar("divideBy", float(b))

    def sum(self) -> float:
        """:467-472"""
        self._require_dense("sum")
        parts = self._all_gather_meta([s.sum() for _, s in self.blocks])
        if not parts:
            raise nat.MarlinError(nat.MB_ERR_EMPTY, "empty collection")
        total = 0.0
        for p in parts:
            total += p
        return total

    def transpose(self) -> "BlockMatrix":
        """:514-523 — per-block materialised transpose, key (r, c) -> (c, r); no data leaves its GPU."""
        self._require_dense("transpose")
        res = [(BlockID(b.column, b.row), s.transpose()) for b, s in self.blocks]
        return BlockMatrix(res, self.numCols(), self.numRows(), self.numBlksByCol(), self.numBlksByRow(),
                           placement=lambda r, c, s=self: s.owner(c, r))

    # ------------------------------------------------------------------ conversions
    def toDenseVecMatrix(self):
        """:575-594 — blocks -> rows.  Rows of block-row r are assembled on owner(r, 0)."""
        from .dense_vec_matrix import DenseVecMatrix
        self._require_dense("toDenseVecMatrix")
        return DenseVecMatrix._from_block_matrix(self)

    def toBlockMatrix(self, newNumByRow: int, newNumByCol: int) -> "BlockMatrix":
        """:610-665 — re-grid.  Pieces are cut as views, shipped once, and pasted into the new blocks."""
        if self._blksByRow == newNumByRow and self._blksByCol == newNumByCol:
            return self
        self._require_dense("toBlockMatrix (re-grid)")
        nr, nc = self.numRows(), self.numCols()
        rl, cl = _ceil_len(nr, self.numBlksByRow()), _ceil_len(nc, self.numBlksByCol())
        nrl, ncl = _ceil_len(nr, newNumByRow), _ceil_len(nc, newNumByCol)
        new_br, new_bc = int(math.ceil(nr / nrl)), int(math.ceil(nc / ncl))
        rank, ws = world()
        new_owner = lambda r, c: comm.elem_owner(r, c, new_bc, ws) if ws > 1 else 0
        local = {(b.row, b.column): s for b, s in self.blocks}
        dt = self._local_dtype()
        dev = Runtime.get().device if Runtime.available() else torch.device("cpu")
        new_blocks: Dict[Tuple[int, int], SubMatrix] = {}
        sends, send_bufs, pastes = [], {}, []
        # intersect every old block with every new block (MTUtils.splitMethod(ranges, newLen), MTUtils.scala:182-202)
        for orow in range(self.numBlksByRow()):
            r_lo, r_hi = orow * rl, min((orow + 1) * rl, nr)
            for ocol in range(self.numBlksByCol()):
                c_lo, c_hi = ocol * cl, min((ocol + 1) * cl, nc)
                src_rank = self.owner(orow, ocol)
                for nrow in range(r_lo // nrl, (r_hi - 1) // nrl + 1):
                    pr0, pr1 = max(r_lo, nrow * nrl), min(r_hi, (nrow + 1) * nrl)
                    for ncol in range(c_lo // ncl, (c_hi - 1) // ncl + 1):
                        pc0, pc1 = max(c_lo, ncol * ncl), min(c_hi, (ncol + 1) * ncl)
                        dst_rank = new_owner(nrow, ncol)
                        key = (orow, ocol, nrow, ncol)
                        piece = None
                        if src_rank == rank:
                            piece = local[(orow, ocol)].slice(pr0 - r_lo, pr1 - r_lo, pc0 - c_lo, pc1 - c_lo)
                        if dst_rank == rank:
                            pastes.append((key, (nrow, ncol), pr0 - nrow * nrl, pr1 - nrow * nrl, pc0 - ncol * ncl,
                                           pc1 - ncol * ncl, piece))
                        if src_rank != dst_rank:
                            sends.append((src_rank, dst_rank, key))
                            if src_rank == rank:
                                packed = piece.copy()
                                send_bufs[key] = packed.buf[: packed.rows * packed.cols]
        shapes = {p[0]: (p[3] - p[2], p[5] - p[4]) for p in pastes}

        def alloc(key):
            r, c = shapes[key]
            return torch.empty(r * c, dtype=dt, device=dev)

        got = comm.exchange(sends, send_bufs, alloc, rank) if ws > 1 else {}
        for key, (nrow, ncol), r0, r1, c0, c1, piece in pastes:
            if (nrow, ncol) not in new_blocks:
                rows = nr - nrow * nrl if (nrow + 1) * nrl > nr else nrl
                cols = nc - ncol * ncl if (ncol + 1) * ncl > nc else ncl
                new_blocks[(nrow, ncol)] = SubMatrix.empty(rows, cols, nat.MB_F64 if dt == torch.float64 else
                                                           (nat.MB_BF16 if dt == torch.bfloat16 else nat.MB_F32), dev)
            if piece is None:
                r, c = shapes[key]
                piece = SubMatrix(buf=got[key], rows=r, cols=c, ld=max(1, r))
            new_blocks[(nrow, ncol)].slice(r0, r1, c0, c1).assign(piece)
        res = [(BlockID(r, c), blk) for (r, c), blk in sorted(new_blocks.items())]
        return BlockMatrix(res, nr, nc, new_br, new_bc)

    # ------------------------------------------------------------------ I/O (next-row (f)-3)
    def saveToFileSystem(self, path: str, format: str = " ") -> None:
        """:550-559 — "blockmatrix": `row-col-rows-cols:v,v,...` column-major; else DenseVecMatrix format."""
        self._require_dense("saveToFileSystem")
        from ..utils.mt_utils import _jdouble
        if format.lower() == "blockmatrix":
            lines = []
            for b, s in self.blocks:
                data = s.toBreeze().reshape(-1, order="F")
                lines.append(f"{b.row}-{b.column}-{s.rows}-{s.cols}:" + ",".join(_jdouble(v) for v in data))
            rank, ws = world()
            import os
            os.makedirs(path, exist_ok=True)
            with open(os.path.join(path, f"part-{rank:05d}"), "w") as fh:
                fh.write("\n".join(lines) + ("\n" if lines else ""))
        else:
            self.toDenseVecMatrix().saveToFileSystem(path)

    def print(self) -> None:
        for b, s in self.blocks[:4]:
            print(f"blockID :[{b.row}, {b.column}], block content below:\n{s.toBreeze()}")
