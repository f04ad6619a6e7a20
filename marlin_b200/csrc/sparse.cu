// Sparse (CSC) blocks on the device: the three products of matrix/SubMatrix.scala:92-100,112-114
// (LibMatrixMult.multDenseSparse / multSparseDense, SparseMatrix.multiply), toDense and SparseMatrix.rand.
//
// Bit-exactness is the contract: every output element is a sequential sum from +0.0 over the reference's term order, each
// term one rounded multiply and one rounded add (__dmul_rn / __dadd_rn never contract into an FMA), and no output is
// written with atomics.  Dense x sparse keeps each output element in a register of one thread.  The two products with a
// sparse left operand scatter a column of A into an output column per step; one warp owns one output column and a
// shared-memory accumulator for a tile of rows, and a __syncwarp between steps puts the terms of each element in order
// (rows within one column of A are distinct, so a step touches each row at most once).
#include "sparse.h"

#include <algorithm>
#include <cstdint>

namespace mb {
namespace {

constexpr int DS_THREADS = 256, DS_RPT = 4, DS_TILE = DS_THREADS * DS_RPT;   // dense x sparse: rows per CTA tile
constexpr int SC_WARPS = 8, SC_TILE = 1024;                                  // scatter products: 8 columns x 1024 rows
constexpr int MAX_GRID_Y = 65535;

// ---- dense A x sparse B: C(r,j) = sum over B's column j in stored order of B(k,j)*A(r,k) (LibMatrixMult.scala:15-41)
__global__ void __launch_bounds__(DS_THREADS) spmm_dense_sparse_kernel(
    const double* __restrict__ A, long long ars, long long acs, int m, const int* __restrict__ bcp,
    const int* __restrict__ bri, const double* __restrict__ bv, double* __restrict__ C, long long crs, long long ccs,
    int accumulate) {
    const long long j = blockIdx.x;
    const int p0 = bcp[j], p1 = bcp[j + 1];
    // :28-29 — a column holding exactly one entry equal to 1.0 copies A's column (so -0.0 survives)
    const bool copy = p1 - p0 == 1 && bv[p0] == 1.0;
    for (int tile = blockIdx.y; (long long)tile * DS_TILE < m; tile += gridDim.y) {
        const int rbase = tile * DS_TILE + threadIdx.x;
        double acc[DS_RPT];
        if (copy) {
            const long long kc = (long long)bri[p0] * acs;
#pragma unroll
            for (int q = 0; q < DS_RPT; ++q) {
                const int r = rbase + q * DS_THREADS;
                acc[q] = r < m ? A[r * ars + kc] : 0.0;
            }
        } else {
#pragma unroll
            for (int q = 0; q < DS_RPT; ++q) acc[q] = 0.0;
            for (int p = p0; p < p1; ++p) {
                const double b = bv[p];
                const double* a = A + (long long)bri[p] * acs;
#pragma unroll
                for (int q = 0; q < DS_RPT; ++q) {
                    const int r = rbase + q * DS_THREADS;
                    if (r < m) acc[q] = __dadd_rn(acc[q], __dmul_rn(b, a[r * ars]));
                }
            }
        }
#pragma unroll
        for (int q = 0; q < DS_RPT; ++q) {
            const int r = rbase + q * DS_THREADS;
            if (r < m) {
                double* c = C + r * crs + j * ccs;
                *c = accumulate ? __dadd_rn(*c, acc[q]) : acc[q];
            }
        }
    }
}

// tp[t*K + k] = first entry of A's column k whose row is >= t*SC_TILE, for t = 0..ntiles (rows are sorted)
__global__ void tile_ptr_kernel(const int* __restrict__ acp, const int* __restrict__ ari, int K, int ntiles,
                                int* __restrict__ tp) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)(ntiles + 1) * K) return;
    const int t = int(i / K), k = int(i % K);
    int lo = acp[k], hi = acp[k + 1];
    const long long bound = (long long)t * SC_TILE;
    while (lo < hi) {
        const int mid = lo + (hi - lo) / 2;
        if (ari[mid] < bound) lo = mid + 1; else hi = mid;
    }
    tp[i] = lo;
}

// ---- sparse A x (dense | sparse) B.  DENSE_B: C(r,j) = sum over k ascending of A(r,k)*B(k,j) where A(r,k) is stored
// (multSparseDense as defined, LibMatrixMult.scala:43-77).  Sparse B: C(r,j) = sum over B's column j in stored order of
// B(k,j)*A(r,k) where A(r,k) is stored (SparseMatrix.multiply, Matrices.scala:122-152).
template <bool DENSE_B>
__global__ void __launch_bounds__(SC_WARPS * 32) spmm_sparse_scatter_kernel(
    const int* __restrict__ acp, const int* __restrict__ ari, const double* __restrict__ av, int m, int K,
    const int* __restrict__ tp, int tile_rows, const double* __restrict__ B, long long brs, long long bcs,
    const int* __restrict__ bcp, const int* __restrict__ bri, const double* __restrict__ bv, int n,
    double* __restrict__ C, long long crs, long long ccs, int accumulate) {
    extern __shared__ double s_acc[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long j = (long long)blockIdx.x * SC_WARPS + warp;
    if (j >= n) return;                                  // warps are independent: no block-wide barrier below
    double* acc = s_acc + warp * tile_rows;
    const int ntiles = (m + tile_rows - 1) / tile_rows;
    const int s0 = DENSE_B ? 0 : bcp[j], s1 = DENSE_B ? K : bcp[j + 1];
    for (int tile = blockIdx.y; tile < ntiles; tile += gridDim.y) {
        const int r0 = tile * tile_rows, rows = min(tile_rows, m - r0);
        for (int r = lane; r < rows; r += 32) acc[r] = 0.0;
        __syncwarp();
        const int* lo_ptr = tp ? tp + (long long)tile * K : acp;
        const int* hi_ptr = tp ? tp + (long long)(tile + 1) * K : acp + 1;
        for (int s = s0; s < s1; ++s) {
            const int k = DENSE_B ? s : bri[s];
            const double b = DENSE_B ? B[k * brs + j * bcs] : bv[s];
            const int lo = lo_ptr[k], hi = hi_ptr[k];
            for (int p = lo + lane; p < hi; p += 32) {
                const int r = ari[p] - r0;
                acc[r] = __dadd_rn(acc[r], __dmul_rn(b, av[p]));
            }
            __syncwarp();
        }
        for (int r = lane; r < rows; r += 32) {
            double* c = C + (long long)(r0 + r) * crs + j * ccs;
            *c = accumulate ? __dadd_rn(*c, acc[r]) : acc[r];
        }
        __syncwarp();
    }
}

// ---- toDense (Matrices.scala:106-119): one warp per column, zeros then the stored entries
__global__ void sparse_to_dense_kernel(const int* __restrict__ cp, const int* __restrict__ ri, const double* __restrict__ v,
                                       int rows, int cols, double* __restrict__ C, long long crs, long long ccs) {
    const long long c = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (c >= cols) return;
    double* col = C + c * ccs;
    for (int r = lane; r < rows; r += 32) col[r * crs] = 0.0;
    __syncwarp();
    for (int p = cp[c] + lane; p < cp[c + 1]; p += 32) col[(long long)ri[p] * crs] = v[p];
}

// ---- SparseMatrix.rand (Matrices.scala:157-173): column c holds `count` distinct rows, sorted, values in [0,1).
// Stream of column c: splitmix64 seeded with mix(seed + golden*(c+1)).  Rows are chosen by selection sampling (Knuth's
// algorithm S): row i is taken when floor(u32 * (rows - i) / 2^32) < count - taken, which takes exactly `count` rows in
// ascending order; each taken row draws its value (top 53 bits * 2^-53) from the same stream.
__host__ __device__ inline unsigned long long sm64_mix(unsigned long long z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
constexpr unsigned long long GOLDEN = 0x9E3779B97F4A7C15ull;

__global__ void sparse_rand_kernel(int rows, int cols, int count, unsigned long long seed, int* __restrict__ cp,
                                   int* __restrict__ ri, double* __restrict__ v) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c > cols) return;
    cp[c] = int(c * count);
    if (c == cols) return;
    unsigned long long state = sm64_mix(seed + GOLDEN * (unsigned long long)(c + 1));
    int taken = 0;
    const long long base = c * count;
    for (int i = 0; i < rows && taken < count; ++i) {
        state += GOLDEN;
        const unsigned long long x = sm64_mix(state);
        if ((((x >> 32) * (unsigned long long)(rows - i)) >> 32) < (unsigned long long)(count - taken)) {
            state += GOLDEN;
            const unsigned long long y = sm64_mix(state);
            ri[base + taken] = i;
            v[base + taken] = double(y >> 11) * 0x1.0p-53;
            ++taken;
        }
    }
}

int tile_rows_for(int m) { return std::min(SC_TILE, ((std::max(m, 1) + 31) / 32) * 32); }
int tiles_for(int m) { return (m + SC_TILE - 1) / SC_TILE; }

template <bool DENSE_B>
cudaError_t launch_scatter(const int* acp, const int* ari, const double* av, int m, int K, const double* B, long long brs,
                           long long bcs, const int* bcp, const int* bri, const double* bv, int n, double* C, long long crs,
                           long long ccs, int accumulate, int* ws, cudaStream_t st, int* launches) {
    if (m == 0 || n == 0) return cudaSuccess;
    const int tile_rows = tile_rows_for(m), ntiles = tiles_for(m);
    const int* tp = nullptr;
    if (ntiles > 1 && K > 0) {
        const long long total = (long long)(ntiles + 1) * K;
        tile_ptr_kernel<<<unsigned((total + 255) / 256), 256, 0, st>>>(acp, ari, K, ntiles, ws);
        ++*launches;
        tp = ws;
    }
    const size_t smem = size_t(SC_WARPS) * tile_rows * sizeof(double);
    // set on every call: the attribute belongs to the current device's context
    cudaError_t e = cudaFuncSetAttribute(spmm_sparse_scatter_kernel<DENSE_B>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         int(SC_WARPS * SC_TILE * sizeof(double)));
    if (e != cudaSuccess) return e;
    dim3 grid(unsigned((n + SC_WARPS - 1) / SC_WARPS), unsigned(std::min(ntiles, MAX_GRID_Y)));
    spmm_sparse_scatter_kernel<DENSE_B><<<grid, SC_WARPS * 32, smem, st>>>(acp, ari, av, m, K, tp, tile_rows, B, brs, bcs, bcp,
                                                                           bri, bv, n, C, crs, ccs, accumulate);
    ++*launches;
    return cudaGetLastError();
}

}  // namespace

long long sparse_tile_ptr_ints(int m, int K) {
    const int ntiles = tiles_for(m);
    return ntiles > 1 ? (long long)(ntiles + 1) * K : 0;
}

cudaError_t spmm_dense_sparse(const double* A, long long ars, long long acs, int m, const int* bcp, const int* bri,
                              const double* bv, int n, double* C, long long crs, long long ccs, int accumulate,
                              cudaStream_t st, int* launches) {
    if (m == 0 || n == 0) return cudaSuccess;
    dim3 grid(unsigned(n), unsigned(std::min((m + DS_TILE - 1) / DS_TILE, MAX_GRID_Y)));
    spmm_dense_sparse_kernel<<<grid, DS_THREADS, 0, st>>>(A, ars, acs, m, bcp, bri, bv, C, crs, ccs, accumulate);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t spmm_sparse_dense(const int* acp, const int* ari, const double* av, int m, int K, const double* B, long long brs,
                              long long bcs, int n, double* C, long long crs, long long ccs, int accumulate, int* ws,
                              cudaStream_t st, int* launches) {
    return launch_scatter<true>(acp, ari, av, m, K, B, brs, bcs, nullptr, nullptr, nullptr, n, C, crs, ccs, accumulate, ws, st,
                                launches);
}

cudaError_t spgemm_to_dense(const int* acp, const int* ari, const double* av, int m, int K, const int* bcp, const int* bri,
                            const double* bv, int n, double* C, long long crs, long long ccs, int accumulate, int* ws,
                            cudaStream_t st, int* launches) {
    return launch_scatter<false>(acp, ari, av, m, K, nullptr, 0, 0, bcp, bri, bv, n, C, crs, ccs, accumulate, ws, st, launches);
}

cudaError_t sparse_to_dense(const int* cp, const int* ri, const double* v, int rows, int cols, double* C, long long crs,
                            long long ccs, cudaStream_t st, int* launches) {
    if (rows == 0 || cols == 0) return cudaSuccess;
    sparse_to_dense_kernel<<<unsigned((cols + 7) / 8), 256, 0, st>>>(cp, ri, v, rows, cols, C, crs, ccs);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t sparse_rand(int rows, int cols, int count, unsigned long long seed, int* cp, int* ri, double* v, cudaStream_t st,
                        int* launches) {
    sparse_rand_kernel<<<unsigned((cols + 1 + 127) / 128), 128, 0, st>>>(rows, cols, count, seed, cp, ri, v);
    ++*launches;
    return cudaGetLastError();
}

}  // namespace mb
