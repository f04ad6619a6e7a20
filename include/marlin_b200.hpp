// marlin_b200.hpp — header-only C++17 host mirror of edu.nju.pasalab.marlin.matrix / .utils for the hot path,
// layered on the C ABI (marlin_b200.h).  The reference is JVM-compiled Scala and no JVM exists in this image, so this
// is the compiled-language host side: same class and method names, argument meaning and error behaviour as the
// reference (`require(...)` -> std::invalid_argument ~ IllegalArgumentException, empty RDD -> std::runtime_error), so
// that tests/cpp/dms_suite.cpp reads like DistributedMatrixSuite.scala.  One process drives one GPU; an
// RDD[(BlockID, SubMatrix)] is a std::vector of pairs.  (The multi-GPU transport lives in the per-rank Python layer,
// marlin_b200/peer.py, on the same C ABI.)
//
// Citations are relative to the reference's src/main/scala/edu/nju/pasalab/marlin/.
#pragma once
#include "marlin_b200.h"

#include <algorithm>
#include <cctype>
#include <cmath>
#include <cstdint>
#include <fstream>
#include <map>
#include <memory>
#include <sstream>
#include <stdexcept>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

namespace marlin {

// ---------------------------------------------------------------------------------------------- errors / context
inline void check(int32_t rc) {
    if (rc == MB_OK) return;
    const std::string msg = mb_last_error();
    if (rc == MB_ERR_INVALID_ARG || rc == MB_ERR_DIM_MISMATCH || rc == MB_ERR_UNSUPPORTED) throw std::invalid_argument(msg);
    throw std::runtime_error(msg);
}

class Context {
public:
    static mb_ctx* get(int device = 0) {
        static Context c(device);
        return c.ctx_;
    }
private:
    explicit Context(int device) { check(mb_init(device, &ctx_)); }      // throws without a B200: no CPU fallback
    ~Context() { mb_shutdown(ctx_); }
    mb_ctx* ctx_ = nullptr;
};

// The executors of one SparkContext on an NVSwitch box: one process per GPU, `world` of them, created collectively with
// the same session string (SURVEY 8e; include/marlin_b200.h section (e)).  A distributed BlockMatrix is, in every
// process, the blocks that process owns plus the GLOBAL dimensions and grid; block (row, col) lives on
// Comm::owner(row, col, blksByCol) = MatrixElemOpPartitioner partition (rdd/MatrixElemOpPartitioner.scala:16) mod world.
class Comm {
public:
    Comm(int rank, int world, const std::string& session) { check(mb_comm_init(Context::get(), rank, world, session.c_str(), &c_)); }
    ~Comm() { if (c_) mb_comm_destroy(c_); }
    Comm(const Comm&) = delete;
    Comm& operator=(const Comm&) = delete;
    int rank() const { return mb_comm_rank(c_); }
    int world() const { return mb_comm_world(c_); }
    void barrier() { check(mb_comm_barrier(c_)); }
    void checkPeers() { check(mb_comm_check(c_)); }          // throws if a device-side wait for a peer ever timed out
    int owner(int row, int col, int blksByCol) const { return mb_elem_partition(row, col, blksByCol) % world(); }
    mb_comm* handle() const { return c_; }
private:
    mb_comm* c_ = nullptr;
};

inline int ceilLen(long total, int parts) { return (int)std::ceil((double)total / (double)parts); }

// A Breeze DenseMatrix[Double] stand-in on the host: column-major.
struct DenseMatrix {
    int rows = 0, cols = 0;
    std::vector<double> data;
    DenseMatrix() = default;
    DenseMatrix(int r, int c) : rows(r), cols(c), data((size_t)r * c, 0.0) {}
    // BDM((a, b), (c, d)) — row-wise literal
    DenseMatrix(std::initializer_list<std::initializer_list<double>> rowsInit) {
        rows = (int)rowsInit.size();
        cols = rows ? (int)rowsInit.begin()->size() : 0;
        data.assign((size_t)rows * cols, 0.0);
        int r = 0;
        for (auto& row : rowsInit) {
            int c = 0;
            for (double v : row) (*this)(r, c++) = v;
            ++r;
        }
    }
    double& operator()(int r, int c) { return data[(size_t)c * rows + r]; }
    double operator()(int r, int c) const { return data[(size_t)c * rows + r]; }
    bool operator==(const DenseMatrix& o) const { return rows == o.rows && cols == o.cols && data == o.data; }
};

// matrix/Block.scala:37-48
struct BlockID {
    int row = 0, column = 0, seq = 0;
    BlockID() = default;
    BlockID(int r, int c, int s = 0) : row(r), column(c), seq(s) {}
    bool operator==(const BlockID& o) const { return row == o.row && column == o.column && seq == o.seq; }
    bool operator<(const BlockID& o) const { return std::tie(row, column, seq) < std::tie(o.row, o.column, o.seq); }
    int hashCode() const { return row * 31 + column + seq; }
};

// ---------------------------------------------------------------------------------------------- SparseMatrix
// matrix/Matrices.scala:136-253 — a CSC block on the device (mb_spblock).  The products return dense blocks.
struct SparseVector {                                                                   // Vectors.sparse(size, indices, values)
    int size = 0;
    std::vector<int32_t> indices;
    std::vector<double> values;
};
class SubMatrix;
class SparseMatrix {
public:
    SparseMatrix() = default;
    SparseMatrix(int numRows, int numCols, const std::vector<SparseVector>& values) {     // one vector per column
        if ((int)values.size() != numCols) throw std::invalid_argument("SparseMatrix: one SparseVector per column");
        std::vector<int32_t> cp(1, 0), ri;
        std::vector<double> v;
        for (const auto& sv : values) {
            if (sv.indices.size() != sv.values.size()) throw std::invalid_argument("SparseVector: indices / values differ in length");
            ri.insert(ri.end(), sv.indices.begin(), sv.indices.end());
            v.insert(v.end(), sv.values.begin(), sv.values.end());
            cp.push_back((int32_t)ri.size());
        }
        *this = fromCSC(numRows, numCols, cp, ri, v);
    }
    static SparseMatrix fromCSC(int numRows, int numCols, const std::vector<int32_t>& colPtr, const std::vector<int32_t>& rowIdx,
                                const std::vector<double>& val) {
        if ((int)colPtr.size() != numCols + 1) throw std::invalid_argument("SparseMatrix: col_ptr needs numCols + 1 entries");
        mb_spblock* h = nullptr;
        check(mb_spblock_upload(Context::get(), numRows, numCols, colPtr.data(), rowIdx.data(), val.data(), &h));
        return SparseMatrix(h);
    }
    // Matrices.scala:236-253 on the device, seeded (see mb_spblock_rand)
    static SparseMatrix rand(int numRows, int numCols, double sparsity, int64_t seed) {
        mb_spblock* h = nullptr;
        check(mb_spblock_rand(Context::get(), numRows, numCols, sparsity, seed, &h));
        return SparseMatrix(h);
    }
    int numRows() const { int32_t r = 0; mb_spblock_info(h_.get(), &r, nullptr, nullptr); return r; }
    int numCols() const { int32_t c = 0; mb_spblock_info(h_.get(), nullptr, &c, nullptr); return c; }
    int64_t nnz() const { int64_t n = 0; mb_spblock_info(h_.get(), nullptr, nullptr, &n); return n; }
    mb_spblock* handle() const { return h_.get(); }
    explicit operator bool() const { return (bool)h_; }
    inline SubMatrix toDense() const;                                                     // :185-198
    inline SubMatrix multiply(const SparseMatrix& o) const;                               // :208-231
    // the scalar ops of SubMatrix.scala:52-58,71-85,121-129: a copy whose stored values are alpha*v + beta (or v / b)
    SparseMatrix mapValues(double alpha, double beta, bool divide = false, double b = 1.0) const {
        mb_spblock* h = nullptr;
        check(mb_spblock_copy(Context::get(), h_.get(), &h));
        SparseMatrix out(h);
        if (nnz() > 0) {
            mb_block *src = nullptr, *dst = nullptr;
            check(mb_spblock_values(Context::get(), h_.get(), &src));
            std::shared_ptr<mb_block> s(src, [](mb_block* p) { mb_block_free(Context::get(), p); });
            check(mb_spblock_values(Context::get(), h, &dst));
            std::shared_ptr<mb_block> d(dst, [](mb_block* p) { mb_block_free(Context::get(), p); });
            check(divide ? mb_block_div(Context::get(), src, b, 0, dst) : mb_block_axpb(Context::get(), src, alpha, beta, dst));
        }
        return out;
    }
private:
    explicit SparseMatrix(mb_spblock* h) : h_(h, [](mb_spblock* p) { mb_spblock_free(Context::get(), p); }) {}
    std::shared_ptr<mb_spblock> h_;
};

// ---------------------------------------------------------------------------------------------- SubMatrix
// matrix/SubMatrix.scala — the per-block value type, device resident: a dense block, or a sparse one (spMatrix).
class SubMatrix {
public:
    SubMatrix() = default;
    explicit SubMatrix(const SparseMatrix& spMatrix) : sp_(spMatrix) {}                 // new SubMatrix(spMatrix = ...)
    explicit SubMatrix(const DenseMatrix& m) {                                        // new SubMatrix(denseMatrix = ...)
        mb_block* b = nullptr;
        check(mb_block_upload(Context::get(), m.data.data(), 0, m.rows, m.cols, std::max(1, m.rows), 0, MB_F64, &b));
        own(b);
    }
    static SubMatrix empty(int rows, int cols) {
        mb_block* b = nullptr;
        check(mb_block_alloc(Context::get(), rows, cols, MB_F64, &b));
        SubMatrix s;
        s.own(b);
        return s;
    }
    // Host fp64 array with Breeze (offset, majorStride, isTranspose) semantics
    static SubMatrix upload(const double* host, long offset, int rows, int cols, int ld, bool isTranspose) {
        mb_block* b = nullptr;
        check(mb_block_upload(Context::get(), host, offset, rows, cols, ld, isTranspose ? 1 : 0, MB_F64, &b));
        SubMatrix s;
        s.own(b);
        return s;
    }
    int rows() const {
        if (sp_) return sp_.numRows();
        int r = 0; mb_block_info(h_.get(), &r, nullptr, nullptr, nullptr, nullptr, nullptr); return r;
    }
    int cols() const {
        if (sp_) return sp_.numCols();
        int c = 0; mb_block_info(h_.get(), nullptr, &c, nullptr, nullptr, nullptr, nullptr); return c;
    }
    bool isSparse() const { return (bool)sp_; }
    const SparseMatrix& sparseBlock() const { return sp_; }
    mb_block* handle() const {
        if (sp_) throw std::invalid_argument("this operation needs a dense block and this block is sparse: convert with toDenseBlocks");
        return h_.get();
    }

    SubMatrix t() const {                                                             // Breeze `.t`: a view
        mb_block* v = nullptr;
        check(mb_block_view_t(Context::get(), h_.get(), &v));
        return view(v);
    }
    SubMatrix slice(int r0, int r1, int c0, int c1) const {                           // m(r0 until r1, c0 until c1): a view
        mb_block* v = nullptr;
        check(mb_block_slice(Context::get(), h_.get(), r0, r1, c0, c1, &v));
        return view(v);
    }
    SubMatrix add(const SubMatrix& o) const { densePair(o, "add"); SubMatrix r = empty(rows(), cols()); check(mb_block_add(Context::get(), h_.get(), o.h_.get(), r.h_.get())); return r; }        // :41-45
    SubMatrix add(double b) const { if (sp_) return SubMatrix(sp_.mapValues(1.0, b)); SubMatrix r = empty(rows(), cols()); check(mb_block_axpb(Context::get(), h_.get(), 1.0, b, r.h_.get())); return r; }                    // :52-58
    SubMatrix subtract(const SubMatrix& o) const { densePair(o, "subtract"); SubMatrix r = empty(rows(), cols()); check(mb_block_sub(Context::get(), h_.get(), o.h_.get(), r.h_.get())); return r; }   // :60-64
    SubMatrix subtract(double b) const { if (sp_) return SubMatrix(sp_.mapValues(1.0, -b)); SubMatrix r = empty(rows(), cols()); check(mb_block_axpb(Context::get(), h_.get(), 1.0, -b, r.h_.get())); return r; }              // :71-77
    SubMatrix divide(double b) const { if (sp_) return SubMatrix(sp_.mapValues(1.0, 0.0, true, b)); SubMatrix r = empty(rows(), cols()); check(mb_block_div(Context::get(), h_.get(), b, 0, r.h_.get())); return r; }                     // :79-85
    SubMatrix multiply(double b) const { if (sp_) return SubMatrix(sp_.mapValues(b, 0.0)); SubMatrix r = empty(rows(), cols()); check(mb_block_axpb(Context::get(), h_.get(), b, 0.0, r.h_.get())); return r; }               // :123-131
    SubMatrix elementMultiply(const SubMatrix& o) const { SubMatrix r = empty(rows(), cols()); check(mb_block_hadamard(Context::get(), h_.get(), o.h_.get(), r.h_.get())); return r; }
    SubMatrix multiply(const SubMatrix& o) const {                                    // :87-91 -> dgemm; sparse arms :92-100
        if (sp_ || o.sp_) {
            SubMatrix r = empty(rows(), o.cols());
            multiplyInto(o, r, false);
            return r;
        }
        if (cols() != o.rows())
            throw std::invalid_argument("Dimension mismatch during matrix-matrix multiplication: " + std::to_string(cols()) + " vs " + std::to_string(o.rows()));
        SubMatrix r = empty(rows(), o.cols());
        check(mb_block_gemm(Context::get(), h_.get(), o.h_.get(), r.h_.get(), 0));
        return r;
    }
    void multiplyInto(const SubMatrix& o, SubMatrix& out, bool accumulate) const {
        const int acc = accumulate ? 1 : 0;
        if (sp_ && o.sp_) check(mb_spgemm_to_dense(Context::get(), sp_.handle(), o.sp_.handle(), out.handle(), acc));          // :92-94
        else if (o.sp_) check(mb_spmm_dense_sparse(Context::get(), handle(), o.sp_.handle(), out.handle(), acc));               // :95-97
        else if (sp_) check(mb_spmm_sparse_dense(Context::get(), sp_.handle(), o.handle(), out.handle(), acc));                 // :98-100
        else check(mb_block_gemm(Context::get(), h_.get(), o.h_.get(), out.h_.get(), acc));
    }
    SubMatrix toDenseBlock() const { return sp_ ? sp_.toDense() : *this; }           // BlockMatrix.scala:598
    SubMatrix transpose() const {                                                     // denseBlock.t.copy (BlockMatrix.scala:517)
        SubMatrix r = empty(cols(), rows());
        check(mb_block_transpose(Context::get(), h_.get(), r.h_.get()));
        return r;
    }
    // vectors are single-column blocks: BDM * BDV goes through multiply() above (dgemv), v.t * w and v * w.t here
    explicit SubMatrix(const std::vector<double>& v) {                                // new DenseVector(array)
        mb_block* b = nullptr;
        if (v.empty()) check(mb_block_alloc(Context::get(), 0, 1, MB_F64, &b));       // an empty piece (more splits than elements)
        else check(mb_block_upload(Context::get(), v.data(), 0, (int)v.size(), 1, (int)v.size(), 0, MB_F64, &b));
        own(b);
    }
    double dot(const SubMatrix& o) const { double d = 0; check(mb_block_dot(Context::get(), h_.get(), o.h_.get(), &d)); return d; }      // DistributedVector.scala:167
    SubMatrix outer(const SubMatrix& o) const {                                       // DistributedVector.scala:157
        SubMatrix r = empty(rows() * cols(), o.rows() * o.cols());
        check(mb_block_ger(Context::get(), h_.get(), o.h_.get(), r.h_.get()));
        return r;
    }
    // brzLU / brzCholesky / brzInv of DenseVecMatrix.luDecompose / choleskyDecompose / inverse (DenseVecMatrix.scala:302,495,587)
    SubMatrix copy() const { SubMatrix r = empty(rows(), cols()); check(mb_block_copy(Context::get(), h_.get(), r.h_.get())); return r; }
    std::pair<SubMatrix, std::vector<int>> lu() const {
        SubMatrix r = copy();
        std::vector<int32_t> perm((size_t)std::max(1, rows()));
        check(mb_block_lu(Context::get(), r.h_.get(), perm.data()));
        return {r, std::vector<int>(perm.begin(), perm.begin() + rows())};
    }
    SubMatrix cholesky() const { SubMatrix r = copy(); check(mb_block_cholesky(Context::get(), r.h_.get())); return r; }
    SubMatrix inverse() const { SubMatrix r = empty(rows(), cols()); check(mb_block_inverse(Context::get(), h_.get(), r.h_.get())); return r; }
    SubMatrix solveTriangular(const SubMatrix& rhs, bool lower, bool unit = false) const {      // this \ rhs
        SubMatrix x = rhs.copy();
        check(mb_block_trsm(Context::get(), h_.get(), lower ? 1 : 0, unit ? 1 : 0, x.h_.get()));
        return x;
    }
    void assign(const SubMatrix& src) { check(mb_block_copy(Context::get(), src.h_.get(), h_.get())); }   // this(range) := src
    double sum() const { double s = 0; check(mb_block_sum(Context::get(), h_.get(), &s)); return s; }
    DenseMatrix denseBlock() const {                                                  // collect to the host (toBreeze)
        if (sp_) return sp_.toDense().denseBlock();
        DenseMatrix m(rows(), cols());
        check(mb_block_download(Context::get(), h_.get(), m.data.data(), std::max(1, m.rows)));
        return m;
    }
private:
    void own(mb_block* b) { h_ = std::shared_ptr<mb_block>(b, [](mb_block* p) { mb_block_free(Context::get(), p); }); }
    SubMatrix view(mb_block* v) const {
        SubMatrix s;
        auto parent = h_;       // a view keeps its parent's storage alive
        s.h_ = std::shared_ptr<mb_block>(v, [parent](mb_block* p) { mb_block_free(Context::get(), p); });
        return s;
    }
    void densePair(const SubMatrix& o, const char* op) const {                      // :46-48, :66-68
        if (sp_ || o.sp_)
            throw std::invalid_argument(std::string("Not supported ") + op + "-operator between matrices of sparsity with " +
                                        (sp_ ? "true" : "false") + " and " + (o.sp_ ? "true" : "false"));
    }
    std::shared_ptr<mb_block> h_;
    SparseMatrix sp_;
};

inline SubMatrix SparseMatrix::toDense() const {
    SubMatrix r = SubMatrix::empty(numRows(), numCols());
    check(mb_spblock_to_dense(Context::get(), h_.get(), r.handle()));
    return r;
}
inline SubMatrix SparseMatrix::multiply(const SparseMatrix& o) const { return SubMatrix(*this).multiply(SubMatrix(o)); }

// matrix/LibMatrixMult.scala
struct LibMatrixMult {
    static SubMatrix multDenseSparse(const SubMatrix& denseMat, const SparseMatrix& sparseMat) {        // :15-41
        return denseMat.multiply(SubMatrix(sparseMat));
    }
    static SubMatrix multSparseDense(const SparseMatrix& sparseMat, const SubMatrix& denseMat) {        // :43-77, as defined
        return SubMatrix(sparseMat).multiply(denseMat);
    }
};

class DenseVecMatrix;
class DistributedVector;

// ---------------------------------------------------------------------------------------------- BlockMatrix
class BlockMatrix {
public:
    using Blocks = std::vector<std::pair<BlockID, SubMatrix>>;
    Blocks blocks;

    BlockMatrix(Blocks b, long nRows = 0, long nCols = 0, int blksByRow = 0, int blksByCol = 0)     // BlockMatrix.scala:28-32
        : blocks(std::move(b)), nRows_(nRows), nCols_(nCols), blksByRow_(blksByRow), blksByCol_(blksByCol) {}

    long numRows() {                                                                  // :36-41
        if (nRows_ <= 0) {
            long s = 0; bool any = false;
            for (auto& kv : blocks) if (kv.first.column == 0) { s += kv.second.rows(); any = true; }
            if (!any) throw std::runtime_error("empty collection");
            nRows_ = s;
        }
        return nRows_;
    }
    long numCols() {                                                                  // :44-49
        if (nCols_ <= 0) {
            long s = 0; bool any = false;
            for (auto& kv : blocks) if (kv.first.row == 0) { s += kv.second.cols(); any = true; }
            if (!any) throw std::runtime_error("empty collection");
            nCols_ = s;
        }
        return nCols_;
    }
    int numBlksByRow() { if (blksByRow_ <= 0) { int n = 0; for (auto& kv : blocks) n += kv.first.column == 0; blksByRow_ = n; } return blksByRow_; }   // :52-57
    int numBlksByCol() { if (blksByCol_ <= 0) { int n = 0; for (auto& kv : blocks) n += kv.first.row == 0; blksByCol_ = n; } return blksByCol_; }     // :60-65
    const Blocks& getBlocks() const { return blocks; }
    long elementsCount() const { return (long)blocks.size(); }                        // :477-479

    DenseMatrix toBreeze() {                                                          // :70-85
        const int m = (int)numRows(), n = (int)numCols();
        const int rl = ceilLen(m, numBlksByRow()), cl = ceilLen(n, numBlksByCol());
        DenseMatrix mat(m, n);
        for (auto& kv : blocks) {
            DenseMatrix b = kv.second.denseBlock();
            for (int c = 0; c < b.cols; ++c)
                for (int r = 0; r < b.rows; ++r) mat(kv.first.row * rl + r, kv.first.column * cl + c) = b(r, c);
        }
        return mat;
    }

    // multiply(other: BlockMatrix) :149-220
    BlockMatrix multiply(BlockMatrix& other) {
        requireMul(numCols(), other.numRows());
        if (numBlksByCol() == other.numBlksByRow()) {
            const int m = numBlksByRow(), k = numBlksByCol(), n = other.numBlksByCol();
            // partition seq = i*n*k + j*k + kk holds A(i,kk) and B(kk,j) (:161-171); on one GPU all m*k*n products and the
            // k-way reduceByKey (:177) run as ONE grouped persistent launch
            std::vector<mb_block*> A((size_t)m * k, nullptr), B((size_t)k * n, nullptr), C((size_t)m * n, nullptr);
            std::map<std::pair<int, int>, SubMatrix> ta, tb;
            for (auto& kv : blocks) { ta[{kv.first.row, kv.first.column}] = kv.second; A[(size_t)kv.first.row * k + kv.first.column] = kv.second.handle(); }
            for (auto& kv : other.blocks) { tb[{kv.first.row, kv.first.column}] = kv.second; B[(size_t)kv.first.row * n + kv.first.column] = kv.second.handle(); }
            Blocks res;
            std::vector<int32_t> ids;
            for (int i = 0; i < m; ++i)
                for (int j = 0; j < n; ++j) {
                    bool complete = true;
                    for (int kk = 0; kk < k; ++kk) complete = complete && A[(size_t)i * k + kk] && B[(size_t)kk * n + j];
                    if (!complete) continue;                                         // the join drops partitions missing a side
                    SubMatrix c = SubMatrix::empty(ta[{i, 0}].rows(), tb[{0, j}].cols());
                    C[(size_t)i * n + j] = c.handle();
                    ids.push_back(i * n + j);
                    res.emplace_back(BlockID(i, j), c);
                }
            if (!ids.empty())
                check(mb_matmul_blocked_subset(Context::get(), A.data(), B.data(), m, k, n, C.data(), ids.data(), (int32_t)ids.size()));
            return BlockMatrix(res, numRows(), other.numCols(), m, n);
        }
        if (numBlksByCol() % other.numBlksByRow() == 0) {                            // :187-201
            checkEvenCols();
            const int ratio = numBlksByCol() / other.numBlksByRow();
            Blocks split;
            for (auto& kv : other.blocks)
                for (int i = 0; i < ratio; ++i) {
                    const int r = kv.second.rows();
                    split.emplace_back(BlockID(kv.first.row * ratio + i, kv.first.column), kv.second.slice(i * r / ratio, (i + 1) * r / ratio, 0, kv.second.cols()));
                }
            BlockMatrix o(split);
            return multiply(o);
        }
        if (other.numBlksByRow() % numBlksByCol() == 0) {                            // :202-216
            checkEvenCols();
            const int ratio = other.numBlksByRow() / numBlksByCol();
            Blocks split;
            for (auto& kv : blocks)
                for (int i = 0; i < ratio; ++i) {
                    const int r = kv.second.rows();
                    split.emplace_back(BlockID(kv.first.row * ratio + i, kv.first.column), kv.second.slice(i * r / ratio, (i + 1) * r / ratio, 0, kv.second.cols()));
                }
            BlockMatrix t(split);
            return t.multiply(other);
        }
        throw std::invalid_argument("currently not supported for the two dimension of matrices");
    }
    // multiply(other: BlockMatrix) :149-186 across the ranks of `comm`: this process passes the blocks it owns (both
    // matrices constructed with their GLOBAL nRows / nCols / grid), and gets back the C blocks mb_dist_plan assigns to it.
    // Replication (:161-171), the block products (:175) and the reduceByKey (:177) all happen inside ONE collective call.
    BlockMatrix multiply(BlockMatrix& other, Comm& comm) {
        if (nRows_ <= 0 || nCols_ <= 0 || blksByRow_ <= 0 || blksByCol_ <= 0 || other.nRows_ <= 0 || other.nCols_ <= 0 ||
            other.blksByRow_ <= 0 || other.blksByCol_ <= 0)
            throw std::invalid_argument("a distributed BlockMatrix needs its global dimensions and grid");
        requireMul(nCols_, other.nRows_);
        if (blksByCol_ != other.blksByRow_) throw std::invalid_argument("currently not supported for the two dimension of matrices");
        const int m = blksByRow_, k = blksByCol_, n = other.blksByCol_, rank = comm.rank();
        auto lens = [](long total, int parts) {                                    // ceil sizing, the last block takes the rest (:73-74)
            std::vector<int32_t> v(parts);
            const int len = ceilLen(total, parts);
            for (int p = 0; p < parts; ++p) v[p] = (int32_t)std::max<long>(0, std::min<long>(len, total - (long)p * len));
            return v;
        };
        const std::vector<int32_t> rowLen = lens(nRows_, m), kLen = lens(nCols_, k), colLen = lens(other.nCols_, n);
        std::vector<mb_block*> A((size_t)m * k, nullptr), B((size_t)k * n, nullptr), C((size_t)m * n, nullptr);
        std::vector<int32_t> aOwner((size_t)m * k), bOwner((size_t)k * n), prodRank((size_t)m * k * n), cOwner((size_t)m * n);
        for (int i = 0; i < m; ++i) for (int kk = 0; kk < k; ++kk) aOwner[(size_t)i * k + kk] = ownerOf(i, kk, comm);
        for (int kk = 0; kk < k; ++kk) for (int j = 0; j < n; ++j) bOwner[(size_t)kk * n + j] = other.ownerOf(kk, j, comm);
        for (auto& kv : blocks) A[(size_t)kv.first.row * k + kv.first.column] = kv.second.handle();
        for (auto& kv : other.blocks) B[(size_t)kv.first.row * n + kv.first.column] = kv.second.handle();
        check(mb_dist_plan(m, k, n, comm.world(), prodRank.data(), cOwner.data()));
        Blocks res;
        for (int i = 0; i < m; ++i)
            for (int j = 0; j < n; ++j)
                if (cOwner[(size_t)i * n + j] == rank) {
                    SubMatrix c = SubMatrix::empty(rowLen[i], colLen[j]);
                    C[(size_t)i * n + j] = c.handle();
                    res.emplace_back(BlockID(i, j), c);
                }
        check(mb_matmul_blocked_dist(comm.handle(), A.data(), aOwner.data(), B.data(), bOwner.data(), m, k, n, rowLen.data(), kLen.data(),
                                     colLen.data(), MB_F64, C.data()));
        BlockMatrix out(res, nRows_, other.nCols_, m, n);
        out.placement_ = cOwner;                 // C(i,j) stays where its kk = 0 partial was computed (no extra move)
        return out;
    }
    // Home rank of block (row, col) of a distributed matrix: MatrixElemOpPartitioner order mod world for matrices built by
    // the caller, the plan's placement for results of a distributed multiply (so products can be chained).
    int ownerOf(int row, int col, const Comm& comm) const {
        return placement_.empty() ? comm.owner(row, col, blksByCol_) : placement_[(size_t)row * blksByCol_ + col];
    }
    // multiply(other, splitMode) :131-147
    BlockMatrix multiply(BlockMatrix& other, std::tuple<int, int, int> splitMode) {
        requireMul(numCols(), other.numRows());
        BlockMatrix a = toBlockMatrix(std::get<0>(splitMode), std::get<1>(splitMode));
        BlockMatrix b = other.toBlockMatrix(std::get<1>(splitMode), std::get<2>(splitMode));
        return a.multiply(b);
    }
    // multiply(other: BlockMatrix, cores, broadcastThreshold = 300) :87-122 (`case that: BlockMatrix`)
    BlockMatrix multiply(BlockMatrix& other, int cores, int broadcastThreshold = 300) {
        requireMul(numCols(), other.numRows());
        int32_t strat = 0, mkn[3] = {0, 0, 0};
        check(mb_choose_strategy(numRows(), numCols(), other.numCols(), cores, broadcastThreshold, 1, &strat, mkn));
        if (strat == 0) return multiply(other.toBreeze());
        if (strat == 1) return other.multiplyBy(toBreeze());
        return multiply(other, std::make_tuple(mkn[0], mkn[1], mkn[2]));
    }
    inline BlockMatrix multiply(DenseVecMatrix& other, int cores, int broadcastThreshold = 300);     // :93-109
    inline DistributedVector multiply(DistributedVector& v);                                         // :240-259
    inline DistributedVector multiply(const std::vector<double>& v);                                 // multiply(v: BDV) :265-274
    BlockMatrix multiply(double b) { return mapBlocks([&](const SubMatrix& s) { return s.multiply(b); }); }     // :229-232
    // multiply(B: BDM[Double]) :280-303
    BlockMatrix multiply(const DenseMatrix& Bm) {
        requireMul(numCols(), Bm.rows);
        SubMatrix B(Bm);
        if (numBlksByCol() == 1) {
            Blocks res;
            for (auto& kv : blocks) res.emplace_back(kv.first, kv.second.multiply(B));
            return BlockMatrix(res, numRows(), Bm.cols, numBlksByRow(), numBlksByCol());
        }
        const int colBlk = ceilLen(numCols(), numBlksByCol());
        std::map<int, SubMatrix> acc;
        Blocks sorted = blocks;
        std::sort(sorted.begin(), sorted.end(), [](auto& a, auto& b) { return a.first < b.first; });
        for (auto& kv : sorted) {
            const int start = kv.first.column * colBlk;
            const int end = (kv.first.column + 1) * colBlk > numCols() ? (int)numCols() : (kv.first.column + 1) * colBlk;
            SubMatrix bs = B.slice(start, end, 0, Bm.cols);
            auto it = acc.find(kv.first.row);
            if (it == acc.end()) acc[kv.first.row] = kv.second.multiply(bs);
            else kv.second.multiplyInto(bs, it->second, true);                       // reduceByKey((a, b) => a.add(b)) fused
        }
        Blocks res;
        for (auto& kv : acc) res.emplace_back(BlockID(kv.first, 0), kv.second);
        return BlockMatrix(res, numRows(), Bm.cols, numBlksByRow(), numBlksByCol());  // (:301 reports numBlksByCol(), kept)
    }
    // multiplyBy(B: BDM[Double]) :309-335 (one block row)
    BlockMatrix multiplyBy(const DenseMatrix& Bm) {
        requireMul(Bm.cols, numRows());
        SubMatrix B(Bm);
        Blocks res;
        if (numBlksByRow() == 1) {
            for (auto& kv : blocks) res.emplace_back(kv.first, B.multiply(kv.second));
        } else {
            const int rowBlk = ceilLen(numRows(), numBlksByRow());
            for (auto& kv : blocks) {
                const int start = kv.first.row * rowBlk;
                int end = (kv.first.row + 1) * rowBlk > numCols() ? (int)numCols() : (kv.first.row + 1) * rowBlk;
                end = std::min(end, Bm.cols);
                res.emplace_back(kv.first, B.slice(0, Bm.rows, start, end).multiply(kv.second));
            }
        }
        return BlockMatrix(res, Bm.rows, numCols(), numBlksByRow(), numBlksByCol());
    }

    BlockMatrix add(double b) { return mapBlocks([&](const SubMatrix& s) { return s.add(b); }); }                 // :368-371
    BlockMatrix subtract(double b) { return mapBlocks([&](const SubMatrix& s) { return s.subtract(b); }); }       // :404-407
    BlockMatrix divide(double b) { return mapBlocks([&](const SubMatrix& s) { return s.divide(b); }); }           // :432-435
    BlockMatrix add(BlockMatrix& o) { return zip(o, [](const SubMatrix& a, const SubMatrix& b) { return a.add(b); }); }                   // :344-360
    BlockMatrix subtract(BlockMatrix& o) { return zip(o, [](const SubMatrix& a, const SubMatrix& b) { return a.subtract(b); }); }         // :380-396
    BlockMatrix dotProduct(BlockMatrix& o) { return zip(o, [](const SubMatrix& a, const SubMatrix& b) { return a.elementMultiply(b); }); } // :486-507
    inline BlockMatrix add(DenseVecMatrix& o);
    inline BlockMatrix subtract(DenseVecMatrix& o);

    double sum() {                                                                    // :467-472
        if (blocks.empty()) throw std::runtime_error("empty collection");
        double s = 0;
        for (auto& kv : blocks) s += kv.second.sum();
        return s;
    }
    BlockMatrix transpose() {                                                         // :514-523
        Blocks res;
        for (auto& kv : blocks) res.emplace_back(BlockID(kv.first.column, kv.first.row), kv.second.transpose());
        return BlockMatrix(res, numCols(), numRows(), numBlksByCol(), numBlksByRow());
    }
    inline DenseVecMatrix toDenseVecMatrix();                                         // :575-594
    // toBlockMatrix(newNumByRow, newNumByCol) :610-665 — pieces cut as views and pasted into the new grid
    BlockMatrix toBlockMatrix(int newByRow, int newByCol) {
        if (blksByRow_ == newByRow && blksByCol_ == newByCol) return *this;
        const int nr = (int)numRows(), nc = (int)numCols();
        const int rl = ceilLen(nr, numBlksByRow()), cl = ceilLen(nc, numBlksByCol());
        const int nrl = ceilLen(nr, newByRow), ncl = ceilLen(nc, newByCol);
        const int newBr = (int)std::ceil((double)nr / nrl), newBc = (int)std::ceil((double)nc / ncl);
        std::map<std::pair<int, int>, SubMatrix> out;
        for (auto& kv : blocks) {
            const int rLo = kv.first.row * rl, rHi = std::min((kv.first.row + 1) * rl, nr);
            const int cLo = kv.first.column * cl, cHi = std::min((kv.first.column + 1) * cl, nc);
            for (int nrow = rLo / nrl; nrow <= (rHi - 1) / nrl; ++nrow)
                for (int ncol = cLo / ncl; ncol <= (cHi - 1) / ncl; ++ncol) {
                    const int r0 = std::max(rLo, nrow * nrl), r1 = std::min(rHi, (nrow + 1) * nrl);
                    const int c0 = std::max(cLo, ncol * ncl), c1 = std::min(cHi, (ncol + 1) * ncl);
                    auto key = std::make_pair(nrow, ncol);
                    if (!out.count(key)) {
                        const int rows = (nrow + 1) * nrl > nr ? nr - nrow * nrl : nrl;
                        const int cols = (ncol + 1) * ncl > nc ? nc - ncol * ncl : ncl;
                        out[key] = SubMatrix::empty(rows, cols);
                    }
                    out[key].slice(r0 - nrow * nrl, r1 - nrow * nrl, c0 - ncol * ncl, c1 - ncol * ncl)
                        .assign(kv.second.slice(r0 - rLo, r1 - rLo, c0 - cLo, c1 - cLo));
                }
        }
        Blocks res;
        for (auto& kv : out) res.emplace_back(BlockID(kv.first.first, kv.first.second), kv.second);
        return BlockMatrix(res, nr, nc, newBr, newBc);
    }

private:
    template <class F> BlockMatrix mapBlocks(F f) {
        Blocks res;
        for (auto& kv : blocks) res.emplace_back(kv.first, f(kv.second));
        return BlockMatrix(res, numRows(), numCols(), numBlksByRow(), numBlksByCol());
    }
    template <class F> BlockMatrix zip(BlockMatrix& o, F f) {
        if (numRows() != o.numRows() || numCols() != o.numCols()) throw std::invalid_argument("matrix dimension mismatch");
        if (numBlksByRow() != o.numBlksByRow() || numBlksByCol() != o.numBlksByCol()) {
            BlockMatrix re = o.toBlockMatrix(numBlksByRow(), numBlksByCol());        // reference goes through DenseVecMatrix (:353-354)
            return zip(re, f);
        }
        std::map<std::pair<int, int>, SubMatrix> theirs;
        for (auto& kv : o.blocks) theirs[{kv.first.row, kv.first.column}] = kv.second;
        Blocks res;
        for (auto& kv : blocks) {
            auto it = theirs.find({kv.first.row, kv.first.column});
            if (it != theirs.end()) res.emplace_back(kv.first, f(kv.second, it->second));    // blocks.join(mat.blocks)
        }
        return BlockMatrix(res, numRows(), numCols(), numBlksByRow(), numBlksByCol());
    }
    static void requireMul(long a, long b) {
        if (a != b) throw std::invalid_argument("Dimension mismatch during matrix-matrix multiplication: " + std::to_string(a) + " vs " + std::to_string(b));
    }
    void checkEvenCols() {
        if (numCols() % numBlksByCol() != 0) throw std::invalid_argument("only supported BlockMatrix which all the sub-matrices have the same cols");
        if ((numCols() / numBlksByCol()) % 2 != 0) throw std::invalid_argument("only supported sub-matrices with even number cols");
    }
    long nRows_, nCols_;
    int blksByRow_, blksByCol_;
    std::vector<int32_t> placement_;             // distributed results only: owner of block (i, j) at [i * blksByCol + j]
};

// ---------------------------------------------------------------------------------------------- DenseVecMatrix
// matrix/DenseVecMatrix.scala — RDD[(Long, BDV[Double])] becomes row ids + ONE row-major device buffer (a transposed
// block view), the matrix the reference packs per partition before its dgemm (:1670-1675).
class DenseVecMatrix {
public:
    using Row = std::pair<long, std::vector<double>>;
    explicit DenseVecMatrix(const std::vector<Row>& rows, long nRows = 0, long nCols = 0) : nRows_(nRows), nCols_(nCols) {
        if (rows.empty()) return;
        const int cols = (int)rows[0].second.size();
        std::vector<double> host((size_t)rows.size() * cols);
        for (size_t i = 0; i < rows.size(); ++i) {
            ids_.push_back(rows[i].first);
            std::copy(rows[i].second.begin(), rows[i].second.end(), host.begin() + i * cols);
        }
        // row-major (n x cols) == the column-major (cols x n) array viewed transposed
        SubMatrix colmajor = SubMatrix::upload(host.data(), 0, cols, (int)rows.size(), std::max(1, cols), false);
        data_ = colmajor.t();
    }
    DenseVecMatrix(std::vector<long> ids, SubMatrix data, long nRows, long nCols) : ids_(std::move(ids)), data_(std::move(data)), nRows_(nRows), nCols_(nCols) {}

    long numCols() { if (nCols_ <= 0) { if (ids_.empty()) throw std::runtime_error("empty collection"); nCols_ = data_.cols(); } return nCols_; }   // :55-61
    long numRows() { if (nRows_ <= 0) { if (ids_.empty()) throw std::runtime_error("empty collection"); nRows_ = *std::max_element(ids_.begin(), ids_.end()) + 1; } return nRows_; }  // :63-69
    const std::vector<long>& rowIds() const { return ids_; }
    const SubMatrix& shard() const { return data_; }

    DenseMatrix toBreeze() {                                                          // :74-84
        DenseMatrix mat((int)numRows(), (int)numCols());
        if (ids_.empty()) return mat;
        DenseMatrix local = data_.denseBlock();
        for (size_t p = 0; p < ids_.size(); ++p)
            for (int c = 0; c < local.cols; ++c) mat((int)ids_[p], c) = local((int)p, c);
        return mat;
    }
    // multiply(B: BDM[Double]) :1660-1680 — one GEMM on the row shard, C rows keep the ids of A rows
    DenseVecMatrix multiply(const DenseMatrix& Bm) {
        if (numCols() != Bm.rows) throw std::invalid_argument("Dimension mismatch during matrix-matrix multiplication: " + std::to_string(numCols()) + " vs " + std::to_string(Bm.rows));
        SubMatrix B(Bm);
        SubMatrix ct = SubMatrix::empty(Bm.cols, (int)ids_.size());                  // column-major (N x rows) == row-major C shard
        SubMatrix c = ct.t();
        data_.multiplyInto(B, c, false);
        return DenseVecMatrix(ids_, c, 0, Bm.cols);
    }
    // multiply(vector: BDV[Double]): BDV[Double] :171-184 — every row dotted with the broadcast vector: one gemv over the
    // row-major shard, results placed by row id
    std::vector<double> multiply(const std::vector<double>& vector) {
        if (ids_.empty()) return {};
        if (data_.cols() != (int)vector.size())
            throw std::invalid_argument("Dimension mismatch during matrix-vector multiplication: " + std::to_string(data_.cols()) + " vs " + std::to_string(vector.size()));
        DenseMatrix y = data_.multiply(SubMatrix(vector)).denseBlock();
        std::vector<double> out(ids_.size(), 0.0);
        for (size_t p = 0; p < ids_.size(); ++p) out.at((size_t)ids_[p]) = y.data[p];
        return out;
    }
    inline DistributedVector multiply(const std::vector<double>& vector, int splitMode);            // :162-165
    inline DistributedVector multiply(DistributedVector& vector, std::pair<int, int> splitMode);    // :149-154
    // multiply(other, splitMode) :109-141 — rows -> blocks (toBlocks) + the seq-keyed block products
    BlockMatrix multiply(DenseVecMatrix& other, std::tuple<int, int, int> splitMode) {
        if (numCols() != other.numRows()) throw std::invalid_argument("Dimension mismatch during matrix-matrix multiplication: " + std::to_string(numCols()) + " vs " + std::to_string(other.numRows()));
        const int m = std::get<0>(splitMode), k = std::get<1>(splitMode), n = std::get<2>(splitMode);
        if (!(m > 0 && k > 0 && n > 0)) throw std::invalid_argument("not supported (m, k, n)");
        BlockMatrix a = toBlockMatrix(m, k), b = other.toBlockMatrix(k, n);
        return a.multiply(b);
    }
    BlockMatrix multiply(BlockMatrix& other, std::tuple<int, int, int> splitMode) {  // :136-139 (re-grids `that` with (m, k), kept)
        BlockMatrix a = toBlockMatrix(std::get<0>(splitMode), std::get<1>(splitMode));
        BlockMatrix b = other.toBlockMatrix(std::get<0>(splitMode), std::get<1>(splitMode));
        return a.multiply(b);
    }
    // multiply(other, cores, broadcastThreshold = 300) :196-231.  Returns a BlockMatrix in the shuffle branch and a
    // DenseVecMatrix in the broadcast branches; C++ needs one type, so the result is handed back as its dense value.
    DenseMatrix multiply(DenseVecMatrix& other, int cores, int broadcastThreshold = 300) {
        if (numCols() != other.numRows()) throw std::invalid_argument("Dimension mismatch during matrix-matrix multiplication: " + std::to_string(numCols()) + " vs " + std::to_string(other.numRows()));
        int32_t strat = 0, mkn[3] = {0, 0, 0};
        check(mb_choose_strategy(numRows(), numCols(), other.numCols(), cores, broadcastThreshold, 0, &strat, mkn));
        if (strat == 0) return multiply(other.toBreeze()).toBreeze();                // :204-205
        if (strat == 1) return other.multiply(toBreeze()).toBreeze();                // :206-207 (operand-order quirk of the reference, kept)
        return multiply(other, std::make_tuple(mkn[0], mkn[1], mkn[2])).toBreeze();
    }
    DenseMatrix multiply(BlockMatrix& other, int cores, int broadcastThreshold = 300) {   // :219-230
        int32_t strat = 0, mkn[3] = {0, 0, 0};
        check(mb_choose_strategy(numRows(), numCols(), other.numCols(), cores, broadcastThreshold, 1, &strat, mkn));
        if (strat == 0) return multiply(other.toBreeze()).toBreeze();
        if (strat == 1) return other.multiplyBy(toBreeze()).toBreeze();
        return multiply(other, std::make_tuple(mkn[0], mkn[1], mkn[2])).toBreeze();
    }
    DenseVecMatrix multiply(double b) { return unary([&](const SubMatrix& s) { return s.multiply(b); }); }      // :853-858
    DenseVecMatrix add(double b) { return unary([&](const SubMatrix& s) { return s.add(b); }); }                // :817-822
    DenseVecMatrix subtract(double b) { return unary([&](const SubMatrix& s) { return s.subtract(b); }); }      // :829-834
    DenseVecMatrix divide(double b) { return unary([&](const SubMatrix& s) { return s.divide(b); }); }          // :866-871
    DenseVecMatrix add(DenseVecMatrix& o) { return binary(o, 0); }                                              // :771-788
    DenseVecMatrix subtract(DenseVecMatrix& o) { return binary(o, 1); }                                         // :795-810
    DenseVecMatrix dotProduct(DenseVecMatrix& o) { return binary(o, 2); }
    DenseVecMatrix add(BlockMatrix& o) { DenseVecMatrix d = o.toDenseVecMatrix(); return add(d); }              // :782-783
    DenseVecMatrix subtract(BlockMatrix& o) { DenseVecMatrix d = o.toDenseVecMatrix(); return subtract(d); }
    DenseVecMatrix dotProduct(BlockMatrix& o) { DenseVecMatrix d = o.toDenseVecMatrix(); return dotProduct(d); }
    double sum() { if (ids_.empty()) throw std::runtime_error("empty collection"); return data_.sum(); }

    BlockMatrix transpose(int numBlocks = 2) {                                        // :1420-1436 (local[2] parallelism)
        BlockMatrix b = toBlockMatrix(std::min(numBlocks, (int)numRows() / 2), 1);
        return b.transpose();
    }
    // toBlockMatrix(numByRow, numByCol) :1259-1328 — runs of consecutive row ids are copied as strided views
    BlockMatrix toBlockMatrix(int numByRow, int numByCol) {
        const int mRows = (int)numRows(), mCols = (int)numCols();
        const int brs = ceilLen(mRows, numByRow), bcs = ceilLen(mCols, numByCol);
        const int byRow = (int)std::ceil((double)mRows / brs), byCol = (int)std::ceil((double)mCols / bcs);
        std::map<std::pair<int, int>, SubMatrix> out;
        size_t p = 0;
        while (p < ids_.size()) {
            size_t q = p + 1;
            const long br = ids_[p] / brs;
            while (q < ids_.size() && ids_[q] == ids_[q - 1] + 1 && ids_[q] / brs == br) ++q;
            const int take = (int)(q - p), r0 = (int)(ids_[p] - br * brs);
            for (int bc = 0; bc < byCol; ++bc) {
                const int c0 = bc * bcs, c1 = std::min((bc + 1) * bcs, mCols);
                auto key = std::make_pair((int)br, bc);
                if (!out.count(key)) {
                    const int rows = br * brs + brs - 1 >= mRows ? mRows - (int)br * brs : brs;
                    const int cols = bc * bcs + bcs - 1 >= mCols ? mCols - bc * bcs : bcs;
                    SubMatrix z = SubMatrix::empty(rows, cols);
                    check(mb_block_fill(Context::get(), z.handle(), 0.0));                         // BDM.zeros (:1318)
                    out[key] = z;
                }
                out[key].slice(r0, r0 + take, 0, c1 - c0).assign(data_.slice((int)p, (int)q, c0, c1));
            }
            p = q;
        }
        BlockMatrix::Blocks res;
        for (auto& kv : out) res.emplace_back(BlockID(kv.first.first, kv.first.second), kv.second);
        return BlockMatrix(res, mRows, mCols, byRow, byCol);
    }
    // toBlocks(m, k, n, mode) :1084-1223 — the blocks of toBlockMatrix keyed with the seq of their target partitions
    std::vector<std::pair<BlockID, SubMatrix>> toBlocks(int m, int k, int n, const std::string& mode) {
        std::string md = mode;
        std::transform(md.begin(), md.end(), md.begin(), ::tolower);
        if (md != "right" && md != "left") throw std::invalid_argument("only 'right' mode or 'left' mode is supported, you should change mode " + mode);
        if (!(m > 0 && k > 0 && n > 0)) throw std::invalid_argument("not supported (m, k, n)");
        std::vector<std::pair<BlockID, SubMatrix>> out;
        if (md == "right") {
            BlockMatrix b = toBlockMatrix(m, k);
            for (auto& kv : b.blocks)
                for (int i = 0; i < n; ++i) out.emplace_back(BlockID(kv.first.row, i, kv.first.row * n * k + i * k + kv.first.column), kv.second);
        } else {
            BlockMatrix b = toBlockMatrix(k, n);
            for (auto& kv : b.blocks)
                for (int i = 0; i < m; ++i) out.emplace_back(BlockID(i, kv.first.column, i * n * k + kv.first.column * k + kv.first.row), kv.second);
        }
        return out;
    }

    // ---- luDecompose / choleskyDecompose / inverse, "breeze" mode (:300-309, :494-497, :585-589): the matrix is one block on
    //      the device and the factorization one library call.  The distributed block algorithms (:310-466, :497-556,
    //      :589-760) live in the Python mirror (marlin_b200/matrix/factorizations.py) on the same block kernels.
    static bool modeIsDist(const std::string& mode, long n) {
        if (mode == "auto") return n > 6000;
        if (mode == "breeze") return false;
        if (mode == "dist") return true;
        throw std::invalid_argument("Do not support mode " + mode + ".");
    }
    SubMatrix asOneBlock() {                                                          // toBreeze() as a device block, rows in id order
        const int n = (int)numRows(), cols = (int)numCols();
        SubMatrix fullT = SubMatrix::empty(cols, n);
        check(mb_block_fill(Context::get(), fullT.handle(), 0.0));
        SubMatrix full = fullT.t();
        for (size_t p = 0; p < ids_.size(); ++p) full.slice((int)ids_[p], (int)ids_[p] + 1, 0, cols).assign(data_.slice((int)p, (int)p + 1, 0, cols));
        return full.copy();
    }
    std::pair<BlockMatrix, std::vector<int>> luDecompose(const std::string& mode = "auto") {
        if (numRows() != numCols()) throw std::invalid_argument("LU decompose only support square matrix: " + std::to_string(numRows()) + " v.s " + std::to_string(numCols()));
        if (modeIsDist(mode, numRows())) throw std::invalid_argument("the C++ mirror runs the local (breeze) mode; use the Python host for mode dist");
        auto res = asOneBlock().lu();
        return {BlockMatrix({{BlockID(0, 0), res.first}}, numRows(), numCols(), 1, 1), res.second};
    }
    BlockMatrix choleskyDecompose(const std::string& mode = "auto") {
        if (numRows() != numCols()) throw std::invalid_argument("LU decompose only support square matrix: " + std::to_string(numRows()) + " v.s " + std::to_string(numCols()));
        if (modeIsDist(mode, numRows())) throw std::invalid_argument("the C++ mirror runs the local (breeze) mode; use the Python host for mode dist");
        return BlockMatrix({{BlockID(0, 0), asOneBlock().cholesky()}}, numRows(), numCols(), 1, 1);
    }
    BlockMatrix inverse(const std::string& mode = "auto") {
        if (numRows() != numCols()) throw std::invalid_argument("Inversion only support square matrix: " + std::to_string(numRows()) + " v.s " + std::to_string(numCols()));
        if (modeIsDist(mode, numRows())) throw std::invalid_argument("the C++ mirror runs the local (breeze) mode; use the Python host for mode dist");
        return BlockMatrix({{BlockID(0, 0), asOneBlock().inverse()}}, numRows(), numCols(), 1, 1);
    }

private:
    template <class F> DenseVecMatrix unary(F f) {
        if (ids_.empty()) return *this;
        // element-wise on the underlying column-major array, re-viewed as the row shard
        return DenseVecMatrix(ids_, f(data_.t()).t(), numRows(), numCols());
    }
    DenseVecMatrix binary(DenseVecMatrix& o, int op) {
        if (numRows() != o.numRows() || numCols() != o.numCols()) throw std::invalid_argument("Dimension mismatch");
        // rows.join(that.rows): line the other matrix's rows up with ours
        std::map<long, int> pos;
        for (size_t p = 0; p < o.ids_.size(); ++p) pos[o.ids_[p]] = (int)p;
        const int n = (int)ids_.size(), cols = (int)numCols();
        SubMatrix alignedT = SubMatrix::empty(cols, n);
        SubMatrix aligned = alignedT.t();
        for (int p = 0; p < n; ++p) aligned.slice(p, p + 1, 0, cols).assign(o.data_.slice(pos.at(ids_[p]), pos.at(ids_[p]) + 1, 0, cols));
        SubMatrix a = data_.t(), b = alignedT;
        SubMatrix r = op == 0 ? a.add(b) : (op == 1 ? a.subtract(b) : a.elementMultiply(b));
        return DenseVecMatrix(ids_, r.t(), numRows(), numCols());
    }
    std::vector<long> ids_;
    SubMatrix data_;
    long nRows_, nCols_;
};

inline DenseVecMatrix BlockMatrix::toDenseVecMatrix() {                               // BlockMatrix.scala:575-594
    const int nr = (int)numRows(), nc = (int)numCols();
    const int rl = ceilLen(nr, numBlksByRow()), cl = ceilLen(nc, numBlksByCol());
    SubMatrix shardT = SubMatrix::empty(nc, nr);
    check(mb_block_fill(Context::get(), shardT.handle(), 0.0));                             // BDV.zeros (:587)
    SubMatrix shard = shardT.t();
    for (auto& kv : blocks)
        shard.slice(kv.first.row * rl, kv.first.row * rl + kv.second.rows(), kv.first.column * cl, kv.first.column * cl + kv.second.cols()).assign(kv.second);
    std::vector<long> ids(nr);
    for (int i = 0; i < nr; ++i) ids[i] = i;
    return DenseVecMatrix(ids, shard, nr, nc);
}
inline BlockMatrix BlockMatrix::add(DenseVecMatrix& o) { BlockMatrix b = o.toBlockMatrix(numBlksByRow(), numBlksByCol()); return add(b); }          // :346-349 (via rows in the reference)
inline BlockMatrix BlockMatrix::subtract(DenseVecMatrix& o) { BlockMatrix b = o.toBlockMatrix(numBlksByRow(), numBlksByCol()); return subtract(b); }
inline BlockMatrix BlockMatrix::multiply(DenseVecMatrix& other, int cores, int broadcastThreshold) {                                              // :93-109
    requireMul(numCols(), other.numRows());
    int32_t strat = 0, mkn[3] = {0, 0, 0};
    check(mb_choose_strategy(numRows(), numCols(), other.numCols(), cores, broadcastThreshold, 0, &strat, mkn));
    if (strat == 0) return multiply(other.toBreeze());
    if (strat == 1) {                                                                 // :97-98 that.multiply(this.toBreeze()) (quirk kept)
        DenseVecMatrix r = other.multiply(toBreeze());
        return r.toBlockMatrix(1, 1);
    }
    BlockMatrix a = toBlockMatrix(mkn[0], mkn[1]), b = other.toBlockMatrix(mkn[1], mkn[2]);
    return a.multiply(b);
}

// ---------------------------------------------------------------------------------------------- DistributedVector
// matrix/DistributedVector.scala — RDD[(Int, DenseVector)] becomes (id, n x 1 block) pairs in HBM.
class DistributedVector {
public:
    using Pieces = std::vector<std::pair<int, SubMatrix>>;
    // (vecId, (oldStart, oldEnd), (newStart, newEnd)) per source partition (:84)
    using SplitStatus = std::vector<std::vector<std::tuple<int, std::pair<int, int>, std::pair<int, int>>>>;
    Pieces vectors;

    explicit DistributedVector(Pieces v, long len = 0, int splits = 0) : vectors(std::move(v)), len_(len), splits_(splits) {}
    explicit DistributedVector(const std::vector<std::pair<int, std::vector<double>>>& host, long len = 0, int splits = 0)
        : len_(len), splits_(splits) {
        for (auto& kv : host) vectors.emplace_back(kv.first, SubMatrix(kv.second));
    }
    bool isColumnMajor() const { return columnMajor_; }
    void setColumnMajor(bool b) { columnMajor_ = b; }
    int splitNum() { if (splits_ <= 0) splits_ = (int)vectors.size(); return splits_; }                 // :31-36
    long length() {                                                                                     // :38-43
        if (len_ <= 0) { long s = 0; for (auto& kv : vectors) s += kv.second.rows(); len_ = s; }
        return len_;
    }
    const Pieces& getVectors() const { return vectors; }

    DistributedVector substract(DistributedVector& v) {                                                 // :45-49 (sic)
        if (length() != v.length())
            throw std::invalid_argument("unsupported vector length: " + std::to_string(length()) + " v.s " + std::to_string(v.length()));
        Pieces res;
        for (auto& a : vectors)
            for (auto& b : v.vectors)
                if (a.first == b.first) res.emplace_back(a.first, a.second.subtract(b.second));
        return DistributedVector(res, v.length(), splitNum());
    }
    DistributedVector transpose() {                                                                     // :56-60
        DistributedVector r(vectors, length(), splitNum());
        r.setColumnMajor(false);
        return r;
    }
    std::vector<double> toBreeze() {                                                                    // :65-73
        std::vector<double> out((size_t)length(), 0.0);
        const long offset = length() / (long)vectors.size();
        for (auto& kv : vectors) {
            DenseMatrix d = kv.second.denseBlock();
            if (kv.first * offset + (long)d.data.size() > (long)out.size()) throw std::out_of_range("slice out of bounds");
            std::copy(d.data.begin(), d.data.end(), out.begin() + kv.first * offset);
        }
        return out;
    }
    DistributedVector toDisVector(const SplitStatus& splitStatusByRow, int splitNum) {                  // :84-107
        const long n = length();
        const int most = ceilLen(n, splitNum);
        Pieces sorted = vectors;
        std::sort(sorted.begin(), sorted.end(), [](auto& a, auto& b) { return a.first < b.first; });
        std::map<int, SubMatrix> out;
        for (size_t pid = 0; pid < splitStatusByRow.size(); ++pid)
            for (auto& st : splitStatusByRow[pid]) {
                const int vecId = std::get<0>(st);
                auto it = out.find(vecId);
                if (it == out.end()) {
                    const int vlen = (long)(vecId + 1) * most > n ? (int)(n - (long)vecId * most) : most;
                    SubMatrix z = SubMatrix::empty(vlen, 1);
                    check(mb_block_fill(Context::get(), z.handle(), 0.0));
                    it = out.emplace(vecId, z).first;
                }
                const auto oldR = std::get<1>(st), newR = std::get<2>(st);
                SubMatrix dst = it->second.slice(newR.first, newR.second + 1, 0, 1);
                dst.assign(sorted[pid].second.slice(oldR.first, oldR.second + 1, 0, 1));
            }
        Pieces res(out.begin(), out.end());
        return DistributedVector(res);
    }
    // Either[Double, BlockMatrix] (:146-180)
    struct Product {
        bool isLeft = false;
        double left = 0.0;
        std::shared_ptr<BlockMatrix> right;
    };
    Product multiply(DistributedVector& other, const std::string& mode = "dist") {
        if (length() != other.length()) throw std::invalid_argument("the length of these two vectors are not the same");
        if (splitNum() != other.splitNum()) throw std::invalid_argument("currently, only support two vectors with the same splits");
        Product p;
        if (columnMajor_ && !other.columnMajor_) {
            BlockMatrix::Blocks blocks;
            for (auto& a : vectors)
                for (auto& b : other.vectors) blocks.emplace_back(BlockID(a.first, b.first), a.second.outer(b.second));
            p.right = std::make_shared<BlockMatrix>(blocks, length(), length(), splitNum(), splitNum());
            return p;
        }
        if (!columnMajor_ && other.columnMajor_) {
            std::string m = mode;
            std::transform(m.begin(), m.end(), m.begin(), [](unsigned char c) { return (char)std::tolower(c); });
            p.isLeft = true;
            if (m == "dist") {
                Pieces sorted = vectors;
                std::sort(sorted.begin(), sorted.end(), [](auto& a, auto& b) { return a.first < b.first; });
                bool any = false;
                for (auto& a : sorted)
                    for (auto& b : other.vectors)
                        if (a.first == b.first) { const double d = a.second.dot(b.second); p.left = any ? p.left + d : d; any = true; }
                if (!any) throw std::runtime_error("empty collection");
                return p;
            }
            if (m == "local") {
                SubMatrix a(toBreeze()), b(other.toBreeze());
                p.left = a.dot(b);
                return p;
            }
            throw std::invalid_argument("unrecognized mode");
        }
        throw std::invalid_argument("the columnMajor status of the two distributed vectors are the same");
    }
    static DistributedVector fromVector(const std::vector<double>& vector, int numSplits) {             // :184-190
        const int vecLen = ceilLen((long)vector.size(), numSplits);
        Pieces pieces;
        for (int i = 0; i < numSplits; ++i) {
            const size_t a = std::min(vector.size(), (size_t)i * vecLen), b = std::min(vector.size(), (size_t)(i + 1) * vecLen);
            pieces.emplace_back(i, SubMatrix(std::vector<double>(vector.begin() + a, vector.begin() + b)));
        }
        return DistributedVector(pieces, (long)vector.size(), numSplits);
    }
private:
    long len_;
    int splits_;
    bool columnMajor_ = true;
};

inline DistributedVector BlockMatrix::multiply(DistributedVector& v) {
    if (numCols() != v.length())
        throw std::invalid_argument("Dimension mismatch during matrix-matrix multiplication " + std::to_string(numCols()) + " v.s " + std::to_string(v.length()));
    if (numBlksByCol() != v.splitNum()) throw std::invalid_argument("not supported matrix or vector");
    std::map<int, SubMatrix> pieces, acc;
    for (auto& kv : v.vectors) pieces[kv.first] = kv.second;
    Blocks sorted = blocks;
    std::sort(sorted.begin(), sorted.end(), [](auto& a, auto& b) { return a.first < b.first; });
    for (auto& kv : sorted) {
        auto it = acc.find(kv.first.row);
        if (it == acc.end()) acc[kv.first.row] = kv.second.multiply(pieces.at(kv.first.column));
        else kv.second.multiplyInto(pieces.at(kv.first.column), it->second, true);     // reduceByKey(add) fused (:251)
    }
    DistributedVector::Pieces res(acc.begin(), acc.end());
    return DistributedVector(res, v.length(), v.splitNum());                           // labelled as the reference does (:252)
}
inline DistributedVector BlockMatrix::multiply(const std::vector<double>& v) {
    if (numCols() != (long)v.size())
        throw std::invalid_argument("matrix columns size " + std::to_string(numCols()) + " not support vector length " + std::to_string(v.size()));
    if (numBlksByCol() != 1) throw std::invalid_argument("should not split the matrix by column");
    SubMatrix x(v);
    DistributedVector::Pieces res;
    Blocks sorted = blocks;
    std::sort(sorted.begin(), sorted.end(), [](auto& a, auto& b) { return a.first < b.first; });
    for (auto& kv : sorted) res.emplace_back(kv.first.row, kv.second.multiply(x));
    return DistributedVector(res, numRows(), numBlksByRow());
}

inline DistributedVector DenseVecMatrix::multiply(const std::vector<double>& vector, int splitMode) {
    BlockMatrix b = toBlockMatrix(splitMode, 1);
    return b.multiply(vector);
}
inline DistributedVector DenseVecMatrix::multiply(DistributedVector& vector, std::pair<int, int> splitMode) {
    if (numCols() != vector.length())
        throw std::invalid_argument("Dimension mismatch during matrix-matrix multiplication: " + std::to_string(numCols()) + " vs " + std::to_string(vector.length()));
    BlockMatrix b = toBlockMatrix(splitMode.first, splitMode.second);
    return b.multiply(vector);
}

// ---------------------------------------------------------------------------------------------- MTUtils
struct MTUtils {
    static std::tuple<int, int, int> splitMethod(long m, long k, long n, int cores) {   // utils/MTUtils.scala:150-175
        int32_t out[3];
        check(mb_choose_split(m, k, n, cores, out));
        return std::make_tuple(out[0], out[1], out[2]);
    }
    static long hashSeed(long seed) { return mb_hash_seed(seed); }                       // :18-21
    // randomDenVecMatrix (:63-73): partition p holds rows [p*N/P, (p+1)*N/P), its own XORShift stream
    static DenseVecMatrix randomDenVecMatrix(long nRows, int nCols, int numPartitions, long seed, double lo = 0.0, double hi = 1.0) {
        std::vector<int64_t> seeds(numPartitions);
        check(mb_partition_seeds(seed, numPartitions, seeds.data()));
        SubMatrix shardT = SubMatrix::empty(nCols, (int)nRows);
        SubMatrix shard = shardT.t();
        long start = 0;
        for (int p = 0; p < numPartitions; ++p) {
            const long end = ((long)(p + 1) * nRows) / numPartitions;
            if (end > start) {
                SubMatrix view = shard.slice((int)start, (int)end, 0, nCols);
                check(mb_fill_uniform(Context::get(), view.handle(), seeds[p], 0, lo, hi, 1));
            }
            start = end;
        }
        std::vector<long> ids(nRows);
        for (long i = 0; i < nRows; ++i) ids[i] = i;
        return DenseVecMatrix(ids, shard, nRows, nCols);
    }
    // randomBlockMatrix (:34-50): one partition per block in row-major BlockID order, column-major fill
    static BlockMatrix randomBlockMatrix(long nRows, long nCols, int numByRow, int numByCol, long seed, double lo = 0.0, double hi = 1.0) {
        const int brs = ceilLen(nRows, numByRow), bcs = ceilLen(nCols, numByCol);
        const int byRow = (int)std::ceil((double)nRows / brs), byCol = (int)std::ceil((double)nCols / bcs);
        std::vector<int64_t> seeds((size_t)byRow * byCol);
        check(mb_partition_seeds(seed, byRow * byCol, seeds.data()));
        BlockMatrix::Blocks blocks;
        for (int idx = 0; idx < byRow * byCol; ++idx) {
            int rows = brs, cols = bcs;
            if (idx >= (byRow - 1) * byCol && (long)brs * byRow > nRows) rows = (int)(nRows - (long)brs * (byRow - 1));
            if ((idx + 1) % byCol == 0 && (long)bcs * byCol > nCols) cols = (int)(nCols - (long)bcs * (byCol - 1));
            SubMatrix blk = SubMatrix::empty(rows, cols);
            check(mb_fill_uniform(Context::get(), blk.handle(), seeds[idx], 0, lo, hi, 0));
            blocks.emplace_back(BlockID(idx / byCol, idx % byCol), blk);
        }
        return BlockMatrix(blocks, nRows, nCols, byRow, byCol);
    }
    // loadMatrixFile (:286-300): `rowIndex:v,v,...`, separators `,\s?|\s+`
    static DenseVecMatrix loadMatrixFile(const std::string& path) {
        if (!(path.rfind("hdfs://", 0) == 0 || path.rfind("tachyon://", 0) == 0 || path.rfind("/", 0) == 0 || path.rfind("~/", 0) == 0))
            throw std::invalid_argument("the path is not in local file System, HDFS or Tachyon");
        std::ifstream in(path);
        if (!in) throw std::runtime_error("cannot open " + path);
        std::vector<DenseVecMatrix::Row> rows;
        std::string line;
        while (std::getline(in, line)) {
            if (line.empty()) continue;
            const size_t colon = line.find(':');
            DenseVecMatrix::Row row;
            row.first = std::stol(line.substr(0, colon));
            std::string body = line.substr(colon + 1);
            for (char& ch : body) if (ch == ',') ch = ' ';
            std::istringstream ss(body);
            double v;
            while (ss >> v) row.second.push_back(v);
            rows.push_back(std::move(row));
        }
        return DenseVecMatrix(rows);
    }
    static DenseVecMatrix arrayToMatrix(const std::vector<std::vector<double>>& array) {   // :402-405
        std::vector<DenseVecMatrix::Row> rows;
        for (size_t i = 0; i < array.size(); ++i) rows.emplace_back((long)i, array[i]);
        return DenseVecMatrix(rows);
    }
};

}  // namespace marlin
