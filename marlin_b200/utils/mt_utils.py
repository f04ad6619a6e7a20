"""MTUtils — the drop-in for edu.nju.pasalab.marlin.utils.MTUtils (utils/MTUtils.scala) on the hot path:
input generators, the split chooser, the text loaders and array conversions.

`sc` (the SparkContext argument of the reference signatures) is accepted and ignored: the "cluster" is the
set of ranks of torch.distributed (one process per GPU).
"""
from __future__ import annotations

import ctypes as C
import math
import os
import re
import time
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from .. import _native as nat
from .. import comm
from ..matrix.block import BlockID
from ..matrix.block_matrix import BlockMatrix
from ..matrix.dense_vec_matrix import DenseVecMatrix
from ..matrix.sparse_matrix import SparseMatrix
from ..matrix.sub_matrix import SubMatrix
from ..runtime import Runtime, world

_SEP = re.compile(r",\s?|\s+")


def _jdouble(v: float) -> str:
    """java.lang.Double.toString: shortest digits that round-trip, plain decimal for 1e-3 <= |v| < 1e7 and computerized
    scientific notation (d.dddE[-]n) outside that range, always at least one digit after the point.  (JDKs before 19
    print a few values with one digit more than the shortest, JDK-4511638; the shortest form is used here.)"""
    v = float(v)
    if v != v:
        return "NaN"
    if v in (float("inf"), float("-inf")):
        return "Infinity" if v > 0 else "-Infinity"
    if v == 0.0:
        return "-0.0" if math.copysign(1.0, v) < 0 else "0.0"
    from decimal import Decimal
    sign, digs, exp = Decimal(repr(abs(v))).as_tuple()
    digits = "".join(str(d) for d in digs).lstrip("0")
    exp += len(digits) - len(digits.rstrip("0"))
    digits = digits.rstrip("0") or "0"
    lead = len(digits) + exp - 1                        # decimal exponent of the leading digit
    neg = "-" if v < 0 else ""
    if 1e-3 <= abs(v) < 1e7:
        if lead >= 0:
            whole = digits[:lead + 1].ljust(lead + 1, "0")
            frac = digits[lead + 1:] or "0"
        else:
            whole, frac = "0", "0" * (-lead - 1) + digits
        return f"{neg}{whole}.{frac}"
    return f"{neg}{digits[0]}.{digits[1:] or '0'}E{lead}"


def _check_path(path: str) -> None:
    if not (path.startswith("hdfs://") or path.startswith("tachyon://") or path.startswith("/") or path.startswith("~/")):
        raise nat.MarlinArgumentError(nat.MB_ERR_INVALID_ARG, "the path is not in local file System, HDFS or Tachyon")


class UniformGenerator:
    """utils/RandomDataGenerator.scala:53-65 — U[start, end) from XORShiftRandom.nextDouble."""

    def __init__(self, start: float = 0.0, end: float = 1.0):
        self.start, self.end = float(start), float(end)


class MTUtils:
    # ------------------------------------------------------------------ seeds / RNG plumbing
    @staticmethod
    def hashSeed(seed: int) -> int:
        """utils/MTUtils.scala:18-21"""
        return int(nat.load().mb_hash_seed(seed))

    @staticmethod
    def _partition_seeds(seed: int, num_partitions: int) -> List[int]:
        out = (C.c_int64 * num_partitions)()
        nat.check(nat.load().mb_partition_seeds(seed, num_partitions, out))
        return [int(v) for v in out]

    @staticmethod
    def _fill(blk: SubMatrix, partition_seed: int, first: int, dist: UniformGenerator, row_major: bool) -> None:
        rt = Runtime.get(); rt.sync_stream()
        nat.check(rt.lib.mb_fill_uniform(rt.ctx, blk.handle(), partition_seed, first, dist.start, dist.end, int(row_major)))

    # ------------------------------------------------------------------ generators
    @staticmethod
    def randomDenVecMatrix(sc, nRows: int, nColumns: int, numPartitions: int = 0,
                           distribution: Optional[UniformGenerator] = None, seed: Optional[int] = None) -> DenseVecMatrix:
        """utils/MTUtils.scala:63-73 -> RandomDenVecRDD (rdd/RandomRDD.scala:161-182).  Partition p holds rows
        [p*N/P, (p+1)*N/P) (:38-41) and is generated on the GPU that owns it (rank p mod G) from the p-th
        nextLong of java.util.Random(seed); values are bit-identical to the reference's XORShift stream for the
        same seed.  The reference's seed is System.nanoTime() and is not exposed (MTUtils.scala:63-73); the extra
        `seed` keyword makes runs reproducible."""
        dist_ = distribution or UniformGenerator(0.0, 1.0)
        rank, ws = world()
        P = numPartitions if numPartitions > 0 else max(ws, 2 if ws == 1 else ws)
        if seed is None:
            seed = time.time_ns()
        seeds = MTUtils._partition_seeds(seed, P)
        rt = Runtime.get()
        shards, ids = [], []
        start = 0
        for p in range(P):
            end = ((p + 1) * nRows) // P
            if p % ws == rank and end > start:
                shards.append((p, start, end))
            start = end
        nloc = sum(e - s for _, s, e in shards)
        buf = torch.empty(nloc * nColumns, dtype=torch.float64, device=rt.device)
        data = SubMatrix(buf=buf, rows=nloc, cols=nColumns, ld=max(1, nColumns), is_transpose=True) if nloc else None
        off = 0
        for p, s, e in shards:
            view = data.slice(off, off + (e - s), 0, nColumns)
            MTUtils._fill(view, seeds[p], 0, dist_, row_major=True)
            ids.append(np.arange(s, e, dtype=np.int64))
            off += e - s
        ids_arr = np.concatenate(ids) if ids else np.zeros(0, dtype=np.int64)
        return DenseVecMatrix(ids=ids_arr, data=data, nRows=nRows, nCols=nColumns)

    @staticmethod
    def randomBlockMatrix(sc, nRows: int, nColumns: int, numByRow: int, numByCol: int, sparseInfo=(False, 1.0),
                          distribution: Optional[UniformGenerator] = None, seed: Optional[int] = None,
                          dtype: int = nat.MB_F64) -> BlockMatrix:
        """utils/MTUtils.scala:34-50 -> RandomBlockRDD (rdd/RandomRDD.scala:184-223): one partition per block in
        row-major BlockID order, `BDM.create(rows, cols, Array.fill(rows*cols)(nextValue()))` (column-major).
        sparseInfo = (True, d): every block is `SparseMatrix.rand(rows, cols, d)` (rdd/RandomRDD.scala:97-100),
        generated on the GPU from the block's partition seed, so a seed reproduces the matrix (the reference's sparse
        generator is unseeded); values are U[0,1) and `distribution` does not apply, as in the reference."""
        sparse, density = bool(sparseInfo[0]), float(sparseInfo[1])
        if sparse and dtype != nat.MB_F64:
            raise nat.MarlinArgumentError(nat.MB_ERR_UNSUPPORTED, "sparse blocks are fp64")
        dist_ = distribution or UniformGenerator(0.0, 1.0)
        brs = int(math.ceil(float(nRows) / float(numByRow)))
        bcs = int(math.ceil(float(nColumns) / float(numByCol)))
        by_row, by_col = int(math.ceil(nRows / brs)), int(math.ceil(nColumns / bcs))
        if seed is None:
            seed = time.time_ns()
        seeds = MTUtils._partition_seeds(seed, by_row * by_col)
        rank, ws = world()
        blocks = []
        for idx in range(by_row * by_col):
            i, j = divmod(idx, by_col)
            if comm.elem_owner(i, j, by_col, ws) != rank:
                continue
            rows = brs
            if idx >= (by_row - 1) * by_col and brs * by_row > nRows:
                rows = nRows - brs * (by_row - 1)
            cols = bcs
            if (idx + 1) % by_col == 0 and bcs * by_col > nColumns:
                cols = nColumns - bcs * (by_col - 1)
            if sparse:
                blocks.append((BlockID(i, j), SubMatrix(spMatrix=SparseMatrix.rand(rows, cols, density, seed=seeds[idx]))))
                continue
            blk = SubMatrix.empty(rows, cols, nat.MB_F64)
            MTUtils._fill(blk, seeds[idx], 0, dist_, row_major=False)
            if dtype != nat.MB_F64:
                blk = blk.copy(dtype)
            blocks.append((BlockID(i, j), blk.mark_ready()))
        return BlockMatrix(blocks, nRows, nColumns, by_row, by_col)

    @staticmethod
    def randomDistVector(sc, length: int, numSplits: int, distribution: Optional[UniformGenerator] = None,
                         seed: Optional[int] = None):
        """utils/MTUtils.scala:86-93 -> RandomDistVectorRDD (rdd/RandomRDD.scala:116-134,103-112): one partition per
        piece, piece i = the first splitLength values of the stream seeded with the i-th nextLong of Random(seed);
        the last piece takes the remainder."""
        from ..matrix.distributed_vector import DistributedVector
        dist_ = distribution or UniformGenerator(0.0, 1.0)
        if seed is None:
            seed = time.time_ns()
        seeds = MTUtils._partition_seeds(seed, numSplits)
        rank, ws = world()
        split_len = int(math.ceil(float(length) / float(numSplits)))
        pieces = []
        for i in range(numSplits):
            if ws > 1 and i % ws != rank:
                continue
            n = length - split_len * i if i == numSplits - 1 else split_len
            blk = SubMatrix.empty(n, 1, nat.MB_F64)
            MTUtils._fill(blk, seeds[i], 0, dist_, row_major=False)
            pieces.append((i, blk))
        return DistributedVector(pieces, length, numSplits)

    @staticmethod
    def onesDistVector(sc, length: int, numSplits: int):
        """utils/MTUtils.scala:128-134 (OnesGenerator pieces)."""
        from ..matrix.distributed_vector import DistributedVector
        rank, ws = world()
        split_len = int(math.ceil(float(length) / float(numSplits)))
        pieces = []
        for i in range(numSplits):
            if ws > 1 and i % ws != rank:
                continue
            n = length - split_len * i if i == numSplits - 1 else split_len
            blk = SubMatrix.zeros(n, 1, nat.MB_F64)
            pieces.append((i, blk.add(1.0)))
        return DistributedVector(pieces)

    # ------------------------------------------------------------------ split chooser
    @staticmethod
    def splitMethod(m: int, k: int, n: int, cores: int) -> Tuple[int, int, int]:
        """utils/MTUtils.scala:150-175"""
        out = (C.c_int32 * 3)()
        nat.check(nat.load().mb_choose_split(m, k, n, cores, out))
        return out[0], out[1], out[2]

    @staticmethod
    def evaluate(mat) -> None:
        """utils/MTUtils.scala:218-220 — force evaluation; here: wait for the GPU."""
        if Runtime.available():
            torch.cuda.synchronize()

    # ------------------------------------------------------------------ conversions
    @staticmethod
    def arrayToMatrix(sc, array: Sequence[Sequence[float]], partitions: int = 2) -> DenseVecMatrix:
        """utils/MTUtils.scala:402-405 — rows are dealt to ranks like sc.parallelize slices."""
        rank, ws = world()
        n = len(array)
        mine = [(i, array[i]) for i in range(n) if ((i * ws) // max(n, 1)) == rank] if ws > 1 else list(enumerate(array))
        return DenseVecMatrix(mine)

    @staticmethod
    def matrixToArray(mat) -> List[List[float]]:
        """utils/MTUtils.scala:416-438"""
        return mat.toBreeze().tolist()

    # ------------------------------------------------------------------ loaders (next-row (f)-3)
    @staticmethod
    def loadMatrixFile(sc, path: str, minPartitions: int = 4) -> DenseVecMatrix:
        """utils/MTUtils.scala:286-300 — `rowIndex:v,v,...`, separators `,\\s?|\\s+`.  Lines are dealt to ranks in
        contiguous chunks (textFile splits)."""
        _check_path(path)
        files = [path] if os.path.isfile(path) else sorted(os.path.join(path, f) for f in os.listdir(path)
                                                           if not f.startswith((".", "_")))
        lines = []
        for f in files:
            with open(f) as fh:
                lines.extend(l.rstrip("\n") for l in fh if l.strip())
        rank, ws = world()
        n = len(lines)
        lo, hi = (rank * n) // ws, ((rank + 1) * n) // ws
        rows = []
        for line in lines[lo:hi]:
            head, body = line.split(":")
            body = body.strip()
            if body.startswith("DenseVector(") and body.endswith(")"):     # what DenseVecMatrix.saveToFileSystem writes
                body = body[len("DenseVector("):-1]
            rows.append((int(head), np.array([float(t) for t in _SEP.split(body) if t != ""], dtype=np.float64)))
        return DenseVecMatrix(rows)

    @staticmethod
    def loadBlockMatrixFile(sc, path: str, minPartitions: int = 4) -> BlockMatrix:
        """utils/MTUtils.scala:324-340 — `row-col-rows-cols:colmajor,...` (the reference requires an hdfs://,
        tachyon:// or file:// prefix here; a plain absolute path is accepted as well)."""
        p = path[len("file://"):] if path.startswith("file://") else path
        files = [p] if os.path.isfile(p) else sorted(os.path.join(p, f) for f in os.listdir(p) if not f.startswith((".", "_")))
        lines = []
        for f in files:
            with open(f) as fh:
                lines.extend(l.strip() for l in fh if l.strip())
        rank, ws = world()
        blocks = []
        for idx, line in enumerate(lines):
            if idx % ws != rank:
                continue
            head, body = line.split(":")
            r, c, nr, nc = (int(t) for t in head.split("-"))
            arr = np.array([float(t) for t in _SEP.split(body) if t != ""], dtype=np.float64).reshape((nr, nc), order="F")
            blocks.append((BlockID(r, c), SubMatrix(arr)))
        placement = None
        if ws > 1:
            import torch.distributed as dist
            keys = [None] * ws
            dist.all_gather_object(keys, [(b.row, b.column) for b, _ in blocks])
            table = {k: r for r, ks in enumerate(keys) for k in ks}
            placement = lambda r, c, t=table: t[(r, c)]
        return BlockMatrix(blocks, placement=placement)
