/* CPU restatement of the reference's sparse block arithmetic (test infrastructure; never linked into the product).
 * Built with -ffp-contract=off: the JVM never fuses a*b+c.  Paths are relative to the reference's
 * src/main/scala/edu/nju/pasalab/marlin/.  Sparse matrices are CSC (col_ptr[cols+1], row_idx, val) — the reference's
 * Array[SparseVector], one vector per column.  Dense matrices are packed column-major with leading dimension ld. */
#include <stdint.h>
#include <string.h>

/* matrix/LibMatrixMult.scala:15-41, literally (the single-1.0-column copy of :28-29 included) */
void sp_mult_dense_sparse(int m, int n, const double* A, int lda, const int* bcp, const int* bri, const double* bv,
                          double* C) {
    memset(C, 0, sizeof(double) * (size_t)m * n);
    for (int i = 0; i < n; ++i) {
        double* c = C + (size_t)i * m;
        const int p0 = bcp[i], len = bcp[i + 1] - bcp[i];
        if (len == 0) continue;
        if (len == 1 && bv[p0] == 1.0) {
            memcpy(c, A + (size_t)bri[p0] * lda, sizeof(double) * m);
        } else {
            for (int k = 0; k < len; ++k)
                for (int j = 0; j < m; ++j) c[j] += bv[p0 + k] * A[(size_t)bri[p0 + k] * lda + j];
        }
    }
}

/* matrix/LibMatrixMult.scala:43-77: the reference's 32x32-blocked loop.  fixed = 1 indexes B as defined
 * (bixi = i*cd + bk); fixed = 0 keeps the reference's `bixi = i*cd + bi` (:60).  Returns -1 (and stops) if the literal
 * loop would read outside B (B is packed: ldb = K). */
int sp_mult_sparse_dense(int m, int K, int n, const int* acp, const int* ari, const double* av, const double* B, double* C,
                         int fixed) {
    memset(C, 0, sizeof(double) * (size_t)m * n);
    const int bs = 32;
    for (int bi = 0; bi < n; bi += bs) {
        for (int bk = 0; bk < K; bk += bs) {
            const int bimin = n < bi + bs ? n : bi + bs;
            const int bklen = (K < bk + bs ? K : bk + bs) - bk;
            for (int i = bi; i < bimin; ++i) {
                const long long bixi = (long long)i * K + (fixed ? bk : bi);
                const long long cixj = (long long)i * m;
                for (int k = 0; k < bklen; ++k) {
                    if (bixi + k >= (long long)K * n) return -1;
                    const double value = B[bixi + k];
                    for (int j = acp[bk + k]; j < acp[bk + k + 1]; ++j) C[cixj + ari[j]] += value * av[j];
                }
            }
        }
    }
    return 0;
}

/* matrix/Matrices.scala:201-231 (SparseMatrix.multiply with vectMultiplyAdd) */
void sp_multiply(int m, int n, const int* acp, const int* ari, const double* av, const int* bcp, const int* bri,
                 const double* bv, double* C) {
    memset(C, 0, sizeof(double) * (size_t)m * n);
    for (int i = 0; i < n; ++i) {
        double* c = C + (size_t)i * m;
        for (int k = bcp[i]; k < bcp[i + 1]; ++k) {
            const int col = bri[k];
            const double bval = bv[k];
            for (int j = acp[col]; j < acp[col + 1]; ++j) c[ari[j]] += bval * av[j];
        }
    }
}

/* matrix/Matrices.scala:185-198 */
void sp_to_dense(int rows, int cols, const int* cp, const int* ri, const double* v, double* C) {
    memset(C, 0, sizeof(double) * (size_t)rows * cols);
    for (int c = 0; c < cols; ++c)
        for (int p = cp[c]; p < cp[c + 1]; ++p) C[(size_t)c * rows + ri[p]] = v[p];
}

/* The seeded SparseMatrix.rand of the product (matrix/Matrices.scala:157-173 with a reproducible stream): column c uses
 * splitmix64 seeded with mix(seed + golden*(c+1)); row i is taken when ((u >> 32) * (rows - i)) >> 32 < count - taken
 * (selection sampling); a taken row's value is (next >> 11) * 2^-53. */
static uint64_t sm64_mix(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

void sp_rand(int rows, int cols, int count, int64_t seed, int* cp, int* ri, double* v) {
    const uint64_t golden = 0x9E3779B97F4A7C15ull;
    for (int c = 0; c <= cols; ++c) cp[c] = c * count;
    for (int c = 0; c < cols; ++c) {
        uint64_t state = sm64_mix((uint64_t)seed + golden * (uint64_t)(c + 1));
        int taken = 0;
        for (int i = 0; i < rows && taken < count; ++i) {
            state += golden;
            const uint64_t x = sm64_mix(state);
            if ((((x >> 32) * (uint64_t)(rows - i)) >> 32) < (uint64_t)(count - taken)) {
                state += golden;
                const uint64_t y = sm64_mix(state);
                ri[(size_t)c * count + taken] = i;
                v[(size_t)c * count + taken] = (double)(y >> 11) * 0x1.0p-53;
                ++taken;
            }
        }
    }
}
