from .block import BlockID
from .block_matrix import BlockMatrix
from .dense_vec_matrix import DenseVecMatrix
from .distributed_matrix import DistributedMatrix
from .distributed_vector import DistributedVector
from .sparse_matrix import LibMatrixMult, SparseMatrix
from .sub_matrix import SubMatrix

__all__ = ["BlockID", "BlockMatrix", "DenseVecMatrix", "DistributedMatrix", "DistributedVector", "LibMatrixMult", "SparseMatrix",
           "SubMatrix"]
