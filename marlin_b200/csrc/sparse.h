#pragma once
#include <cuda_runtime.h>

namespace mb {

// Sparse blocks are CSC (matrix/Matrices.scala:57-104, one SparseVector per column): col_ptr[cols+1], row_idx[nnz] strictly
// increasing within a column, val[nnz].  Dense operands are views: element (r,c) at base[r*rs + c*cs].
// Every product writes each output element as a sequential sum from +0.0 in the reference's order, one rounded multiply
// and one rounded add per term (no FMA, no atomics); accumulate adds the finished sum to the output with one rounding.

// C = A (m x K dense) * B (K x n CSC)   (LibMatrixMult.multDenseSparse)
cudaError_t spmm_dense_sparse(const double* A, long long ars, long long acs, int m, const int* bcp, const int* bri,
                              const double* bv, int n, double* C, long long crs, long long ccs, int accumulate,
                              cudaStream_t st, int* launches);
// C = A (m x K CSC) * B (K x n dense)   (LibMatrixMult.multSparseDense, as defined: k ascending)
// C = A (m x K CSC) * B (K x n CSC)     (SparseMatrix.multiply)
// Both need a workspace of sparse_tile_ptr_ints(m, K) ints (nullptr when that is 0).
long long sparse_tile_ptr_ints(int m, int K);
cudaError_t spmm_sparse_dense(const int* acp, const int* ari, const double* av, int m, int K, const double* B, long long brs,
                              long long bcs, int n, double* C, long long crs, long long ccs, int accumulate, int* ws,
                              cudaStream_t st, int* launches);
cudaError_t spgemm_to_dense(const int* acp, const int* ari, const double* av, int m, int K, const int* bcp, const int* bri,
                            const double* bv, int n, double* C, long long crs, long long ccs, int accumulate, int* ws,
                            cudaStream_t st, int* launches);
// C (rows x cols view) = toDense of the CSC block (Matrices.scala:106-119)
cudaError_t sparse_to_dense(const int* cp, const int* ri, const double* v, int rows, int cols, double* C, long long crs,
                            long long ccs, cudaStream_t st, int* launches);
// SparseMatrix.rand layout: `count` distinct sorted rows per column from the column's own stream of `seed`
cudaError_t sparse_rand(int rows, int cols, int count, unsigned long long seed, int* cp, int* ri, double* v, cudaStream_t st,
                        int* launches);

}  // namespace mb
