"""marlin_b200 — B200-native engine for the dense block-matrix hot path of PasaLab/marlin.

Public surface mirrors edu.nju.pasalab.marlin.{matrix,utils,rdd} for that path only:
BlockMatrix / DenseVecMatrix / DistributedVector / SubMatrix (dense or sparse) / SparseMatrix / LibMatrixMult / BlockID, MTUtils, MatrixMultPartitioner /
MatrixElemOpPartitioner.  All arithmetic runs in libmarlin_b200.so (hand-written sm_100a kernels).
"""
import os as _os

# One hardware queue per stream: the multi-GPU engine orders its copy / compute / download streams through flags in
# device memory, which the driver cannot see — streams that share a queue could be serialised in the wrong order.
# Only effective if it is set before the CUDA context exists (import marlin_b200 before the first CUDA call).
_os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

from ._native import MarlinArgumentError, MarlinError
from .matrix import (BlockID, BlockMatrix, DenseVecMatrix, DistributedMatrix, DistributedVector, LibMatrixMult, SparseMatrix,
                     SubMatrix)
from .rdd import MatrixElemOpPartitioner, MatrixMultPartitioner
from .runtime import Runtime
from .utils import MTUtils

__all__ = ["BlockID", "BlockMatrix", "DenseVecMatrix", "DistributedMatrix", "DistributedVector", "SubMatrix", "SparseMatrix",
           "LibMatrixMult", "MTUtils",
           "MatrixElemOpPartitioner", "MatrixMultPartitioner", "Runtime", "MarlinError", "MarlinArgumentError"]
