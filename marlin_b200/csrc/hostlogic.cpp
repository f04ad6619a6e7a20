// Pure integer host logic of the multiply path, exported through the C ABI.
// Each function cites the reference code it mirrors (src/main/scala/edu/nju/pasalab/marlin/...).
#include "../../include/marlin_b200.h"
#include <cmath>
#include <cstdint>
#include <cstring>

int32_t mb_fail(int32_t code, const char* fmt, ...);   // capi.cu: sets mb_last_error()

namespace {

// utils/MTUtils.scala:204-213
int dim_to_split(int64_t m, int64_t k, int64_t n) {
    if (n >= k && n >= m) return 1;
    if (m >= k && m >= n) return 2;
    return 3;
}

inline uint32_t rotl32(uint32_t x, int r) { return (x << r) | (x >> (32 - r)); }

// scala.util.hashing.MurmurHash3 (Scala 2.10 library, not in the reference tree): mix / mixLast /
// finalizeHash and bytesHash(data, arraySeed = 0x3c074a61).
uint32_t mm3_mix_last(uint32_t h, uint32_t k) {
    k *= 0xcc9e2d51u;
    k = rotl32(k, 15);
    k *= 0x1b873593u;
    return h ^ k;
}
uint32_t mm3_mix(uint32_t h, uint32_t k) {
    h = mm3_mix_last(h, k);
    h = rotl32(h, 13);
    return h * 5u + 0xe6546b64u;
}
uint32_t mm3_finalize(uint32_t h, uint32_t len) {
    h ^= len;
    h ^= h >> 16;
    h *= 0x85ebca6bu;
    h ^= h >> 13;
    h *= 0xc2b2ae35u;
    h ^= h >> 16;
    return h;
}
uint32_t mm3_bytes_hash(const uint8_t* data, int len, uint32_t seed) {
    uint32_t h = seed;
    int i = 0, rem = len;
    while (rem >= 4) {
        uint32_t k = data[i] | (uint32_t(data[i + 1]) << 8) | (uint32_t(data[i + 2]) << 16) | (uint32_t(data[i + 3]) << 24);
        h = mm3_mix(h, k);
        i += 4;
        rem -= 4;
    }
    uint32_t k = 0;
    if (rem == 3) k ^= uint32_t(data[i + 2]) << 16;
    if (rem >= 2) k ^= uint32_t(data[i + 1]) << 8;
    if (rem >= 1) {
        k ^= data[i];
        h = mm3_mix_last(h, k);
    }
    return mm3_finalize(h, uint32_t(len));
}

}  // namespace

extern "C" {

// utils/MTUtils.scala:150-175 — CARMA-style halving of the largest dimension while cores remain.
int32_t mb_choose_split(int64_t m, int64_t k, int64_t n, int32_t cores, int32_t out_mkn[3]) {
    if (!out_mkn) return MB_ERR_INVALID_ARG;
    int ms = 1, ks = 1, ns = 1;
    int64_t _m = m, _k = k, _n = n;
    int c = cores;
    while (c > 1 && _m > 1 && _k > 1 && _n > 1) {
        const int d = dim_to_split(_m, _k, _n);
        if (d == 1) { ns *= 2; _n /= 2; }
        else if (d == 2) { ms *= 2; _m /= 2; }
        else { ks *= 2; _k /= 2; }
        c /= 2;
    }
    out_mkn[0] = ms; out_mkn[1] = ks; out_mkn[2] = ns;
    return MB_OK;
}

// matrix/DenseVecMatrix.scala:196-231 and matrix/BlockMatrix.scala:87-122.
// broadcastSize = threshold*1024*1024/8 is evaluated in Int arithmetic in the reference.
int32_t mb_choose_strategy(int64_t a_rows, int64_t a_cols, int64_t b_cols, int32_t cores,
                           int32_t broadcast_threshold_mb, int32_t other_is_block, int32_t* strategy,
                           int32_t out_mkn[3]) {
    if (!strategy || !out_mkn) return MB_ERR_INVALID_ARG;
    const int32_t broadcast_size = int32_t(uint32_t(broadcast_threshold_mb) * 1024u * 1024u) / 8;  // JVM Int wrap-around
    const int64_t b_rows = a_cols;
    out_mkn[0] = out_mkn[1] = out_mkn[2] = 0;
    if (b_rows * b_cols <= broadcast_size) { *strategy = 0; return MB_OK; }
    if (a_rows * a_cols <= broadcast_size) { *strategy = 1; return MB_OK; }
    *strategy = 2;
    if (!other_is_block) {
        // `numRows() / numCols()` is Long integer division in the reference (DenseVecMatrix.scala:210-211),
        // so the last two tests read 0.8 < floor(M/K) < 1.2, i.e. floor(M/K) == 1.
        const double ratio = double(a_rows * b_cols) / double(a_cols * a_cols);
        const int64_t q = a_cols ? a_rows / a_cols : 0;
        if (0.8 < ratio && ratio < 1.2 && double(q) < 1.2 && double(q) > 0.8) {
            const int split = int(std::floor(std::pow(3.0 * cores, 1.0 / 3.0)));
            out_mkn[0] = out_mkn[1] = out_mkn[2] = split;
            return MB_OK;
        }
    }
    return mb_choose_split(a_rows, a_cols, b_cols, cores, out_mkn);
}

// rdd/MatrixMultPartitioner.scala:12-22 with seq from matrix/BlockMatrix.scala:163,168
int32_t mb_mult_partition(int32_t i, int32_t j, int32_t kk, int32_t m, int32_t k, int32_t n) {
    (void)m;
    return i * n * k + j * k + kk;
}

// rdd/MatrixElemOpPartitioner.scala:16
int32_t mb_elem_partition(int32_t row, int32_t col, int32_t blks_by_col) { return row * blks_by_col + col; }

// matrix/BlockMatrix.scala:73-74; matrix/DenseVecMatrix.scala:1091-1094,1262-1265
int32_t mb_block_len(int64_t total, int32_t parts, int32_t* block_len, int32_t* actual_parts) {
    if (parts <= 0 || total <= 0 || !block_len || !actual_parts) return MB_ERR_INVALID_ARG;
    const int32_t len = int32_t(std::ceil(double(total) / double(parts)));
    *block_len = len;
    *actual_parts = int32_t(std::ceil(double(total) / double(len)));
    return MB_OK;
}

// utils/MTUtils.scala:18-21: ByteBuffer.allocate(java.lang.Long.SIZE /* = 64 bytes */).putLong(seed)
// -> MurmurHash3.bytesHash -> Int, widened (sign-extended) to Long.
int64_t mb_hash_seed(int64_t seed) {
    uint8_t buf[64];
    std::memset(buf, 0, sizeof(buf));
    for (int i = 0; i < 8; ++i) buf[i] = uint8_t(uint64_t(seed) >> (56 - 8 * i));   // big-endian putLong
    return int64_t(int32_t(mm3_bytes_hash(buf, 64, 0x3c074a61u)));
}

// rdd/RandomRDD.scala:28-45: partition i gets java.util.Random(seed).nextLong() (i-th draw).
int32_t mb_partition_seeds(int64_t seed, int32_t num_partitions, int64_t* seeds_out) {
    if (num_partitions < 0 || (num_partitions > 0 && !seeds_out)) return MB_ERR_INVALID_ARG;
    const uint64_t mask = (1ull << 48) - 1;
    uint64_t s = (uint64_t(seed) ^ 0x5DEECE66Dull) & mask;
    auto next32 = [&]() -> int32_t {
        s = (s * 0x5DEECE66Dull + 0xBull) & mask;
        return int32_t(s >> 16);
    };
    for (int i = 0; i < num_partitions; ++i) {
        const int64_t hi = int64_t(next32());
        const int64_t lo = int64_t(next32());
        seeds_out[i] = int64_t((uint64_t(hi) << 32) + uint64_t(lo));   // ((long)next(32) << 32) + next(32)
    }
    return MB_OK;
}

// matrix/Matrices.scala:57-104 (SparseMatrix as one SparseVector per column) as CSC.  Checked before any upload.
int32_t mb_csc_check(int32_t rows, int32_t cols, const int32_t* col_ptr, const int32_t* row_idx) {
    if (rows < 0 || cols < 0) return mb_fail(MB_ERR_INVALID_ARG, "sparse block: negative dimension %d x %d", rows, cols);
    if (!col_ptr) return mb_fail(MB_ERR_INVALID_ARG, "sparse block: null col_ptr");
    if (col_ptr[0] != 0) return mb_fail(MB_ERR_INVALID_ARG, "sparse block: col_ptr[0] = %d, expected 0", col_ptr[0]);
    for (int32_t c = 0; c < cols; ++c)
        if (col_ptr[c + 1] < col_ptr[c])
            return mb_fail(MB_ERR_INVALID_ARG, "sparse block: col_ptr decreases at column %d (%d > %d)", c, col_ptr[c],
                           col_ptr[c + 1]);
    if (col_ptr[cols] > 0 && !row_idx) return mb_fail(MB_ERR_INVALID_ARG, "sparse block: null row_idx");
    for (int32_t c = 0; c < cols; ++c) {
        for (int32_t p = col_ptr[c]; p < col_ptr[c + 1]; ++p) {
            if (row_idx[p] < 0 || row_idx[p] >= rows)
                return mb_fail(MB_ERR_INVALID_ARG, "sparse block: row index %d of column %d outside [0, %d)", row_idx[p], c, rows);
            if (p > col_ptr[c] && row_idx[p] <= row_idx[p - 1])
                return mb_fail(MB_ERR_INVALID_ARG, "sparse block: row indices of column %d not strictly increasing (%d after %d)",
                               c, row_idx[p], row_idx[p - 1]);
        }
    }
    return MB_OK;
}

// matrix/Matrices.scala:157-173: sparseSize = (numCols * sparsity).toInt
int32_t mb_sparse_rand_count(int32_t rows, int32_t cols, double sparsity, int32_t* count) {
    if (!count || rows < 0 || cols < 0) return mb_fail(MB_ERR_INVALID_ARG, "SparseMatrix.rand: bad argument");
    if (!(sparsity >= 0.0)) return mb_fail(MB_ERR_INVALID_ARG, "SparseMatrix.rand: sparsity %g must be >= 0", sparsity);
    const double want = double(cols) * sparsity;
    if (want >= 2147483648.0) return mb_fail(MB_ERR_INVALID_ARG, "SparseMatrix.rand: %g entries per column", want);
    const int32_t s = int32_t(want);
    if (s > rows)
        return mb_fail(MB_ERR_INVALID_ARG, "SparseMatrix.rand: %d distinct rows per column requested from %d rows", s, rows);
    if (int64_t(s) * cols >= (int64_t(1) << 31))
        return mb_fail(MB_ERR_INVALID_ARG, "SparseMatrix.rand: %lld entries, larger than Int.MaxValue", (long long)s * cols);
    *count = s;
    return MB_OK;
}

}  // extern "C"
