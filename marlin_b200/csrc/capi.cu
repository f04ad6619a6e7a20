// C ABI of libmarlin_b200.so (see include/marlin_b200.h).  Context, block handles and dispatch.
// There is no CPU fallback anywhere in this file: without a CUDA device mb_init fails with
// MB_ERR_CUDA and no compute entry can be reached.
#include "../../include/marlin_b200.h"
#include "elementwise.h"
#include "gemm_f64.h"
#include "gemm_bf16.h"
#include "gemm_ozaki.h"
#include "blas12.h"
#include "factor.h"
#include "sparse.h"

#include <cuda_runtime.h>
#include <algorithm>
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <new>
#include <atomic>
#include <mutex>
#include <vector>

#include "internal.h"

namespace {

thread_local char g_err[512] = "";

int32_t new_block(mb_block** out) {
    *out = new (std::nothrow) mb_block();
    if (!*out) return fail(MB_ERR_OOM, "host allocation failed");
    return MB_OK;
}

int32_t same_shape(const mb_block* a, const mb_block* b, const char* what) {
    if (a->rows != b->rows || a->cols != b->cols)
        return fail(MB_ERR_DIM_MISMATCH, "matrix dimension mismatch in %s: %dx%d vs %dx%d", what, a->rows, a->cols,
                    b->rows, b->cols);
    return MB_OK;
}

int32_t binary_op(mb_ctx* ctx, int op, const mb_block* A, const mb_block* B, mb_block* out, const char* name) {
    MB_CTX(ctx);
    if (!A || !B || !out) return fail(MB_ERR_INVALID_ARG, "%s: null block", name);
    int32_t r = same_shape(A, B, name);
    if (r) return r;
    r = same_shape(A, out, name);
    if (r) return r;
    const bool all_f32 = A->dtype == MB_F32 && B->dtype == MB_F32 && out->dtype == MB_F32;
    if (!all_f32 && (A->dtype != MB_F64 || B->dtype != MB_F64 || out->dtype != MB_F64))
        return fail(MB_ERR_UNSUPPORTED, "%s: fp64 (or all-fp32) blocks only (convert bf16 blocks with mb_block_copy)", name);
    // iterate in the output's storage order so the store side is contiguous
    int rows = A->rows, cols = A->cols;
    long long ars = rs(A), acs = cs(A), brs = rs(B), bcs = cs(B), ors = rs(out), ocs = cs(out);
    if (out->is_transpose) {
        std::swap(rows, cols);
        std::swap(ars, acs); std::swap(brs, bcs); std::swap(ors, ocs);
    }
    if (all_f32) {
        MB_CUDA(mb::ew_binary_f32(op, rows, cols, reinterpret_cast<const float*>(elem_ptr(A)), ars, acs,
                                  reinterpret_cast<const float*>(elem_ptr(B)), brs, bcs, reinterpret_cast<float*>(elem_ptr(out)), ors,
                                  ocs, ctx->stream));
        ctx->launches++;
        return MB_OK;
    }
    MB_CUDA(mb::ew_binary(op, rows, cols, f64_ptr(A), ars, acs, f64_ptr(B), brs, bcs, f64_ptr(out), ors, ocs, ctx->stream));
    ctx->launches++;
    return MB_OK;
}

int32_t unary_op(mb_ctx* ctx, int op, const mb_block* A, mb_block* out, double alpha, double beta, const char* name) {
    MB_CTX(ctx);
    if (!A || !out) return fail(MB_ERR_INVALID_ARG, "%s: null block", name);
    int32_t r = same_shape(A, out, name);
    if (r) return r;
    if (A->dtype != MB_F64 || out->dtype != MB_F64)
        return fail(MB_ERR_UNSUPPORTED, "%s: fp64 blocks only", name);
    int rows = A->rows, cols = A->cols;
    long long ars = rs(A), acs = cs(A), ors = rs(out), ocs = cs(out);
    if (out->is_transpose) {
        std::swap(rows, cols);
        std::swap(ars, acs); std::swap(ors, ocs);
    }
    MB_CUDA(mb::ew_unary(op, rows, cols, f64_ptr(A), ars, acs, f64_ptr(out), ors, ocs, alpha, beta, ctx->stream));
    ctx->launches++;
    return MB_OK;
}

// out (col-major packed or strided, same logical shape as `A` view) = A, with dtype conversion.
int32_t copy_convert(mb_ctx* ctx, const mb_block* A, mb_block* out) {
    int rows = A->rows, cols = A->cols;
    long long ars = rs(A), acs = cs(A), ors = rs(out), ocs = cs(out);
    if (out->is_transpose) {
        std::swap(rows, cols);
        std::swap(ars, acs); std::swap(ors, ocs);
    }
    if (A->dtype == MB_F64 && out->dtype == MB_F64) {
        if (ars == 1 && ors == 1) {
            MB_CUDA(mb::ew_unary(mb::EW_COPY, rows, cols, f64_ptr(A), ars, acs, f64_ptr(out), ors, ocs, 1.0, 0.0, ctx->stream));
        } else if (acs == 1 && ors == 1) {
            // source is the transpose of a column-major (cols x rows, ld = ars) array
            MB_CUDA(mb::transpose_f64(f64_ptr(A), ars, f64_ptr(out), ocs, cols, rows, ctx->stream));
        } else {
            MB_CUDA(mb::ew_unary(mb::EW_COPY, rows, cols, f64_ptr(A), ars, acs, f64_ptr(out), ors, ocs, 1.0, 0.0, ctx->stream));
        }
    } else if (A->dtype == out->dtype && acs == 1 && ors == 1 && A->dtype == MB_BF16) {
        MB_CUDA(mb::transpose_b16(elem_ptr(A), ars, elem_ptr(out), ocs, cols, rows, ctx->stream));
    } else if (A->dtype == out->dtype && acs == 1 && ors == 1 && A->dtype == MB_F32) {
        MB_CUDA(mb::transpose_b32(elem_ptr(A), ars, elem_ptr(out), ocs, cols, rows, ctx->stream));
    } else {
        MB_CUDA(mb::convert_strided(A->dtype, out->dtype, rows, cols, elem_ptr(A), ars, acs, elem_ptr(out), ors, ocs, ctx->stream));
    }
    ctx->launches++;
    return MB_OK;
}


// A block with one column (or one row) read as a vector: element i lives at p[i * inc].
struct vec_view {
    double* p;
    long long inc;
    int len;
};
bool as_vector(const mb_block* b, vec_view* v) {
    if (b->dtype != MB_F64) return false;
    if (b->cols == 1) { v->len = b->rows; v->inc = rs(b); }
    else if (b->rows == 1) { v->len = b->cols; v->inc = cs(b); }
    else return false;
    v->p = f64_ptr(b);
    return true;
}

}  // namespace

int32_t mb_fail(int32_t code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

extern "C" {

const char* mb_last_error(void) { return g_err; }
const char* mb_version(void) { return "marlin_b200 0.1 (sm_100a)"; }

int32_t mb_init(int32_t device, mb_ctx** out) {
    if (!out) return fail(MB_ERR_INVALID_ARG, "mb_init: null out");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(MB_ERR_CUDA, "mb_init: no CUDA device (%s); marlin_b200 has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= count) return fail(MB_ERR_INVALID_ARG, "mb_init: device %d out of range [0,%d)", device, count);
    MB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    MB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(MB_ERR_UNSUPPORTED, "mb_init: device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);
    mb_ctx* ctx = new (std::nothrow) mb_ctx();
    if (!ctx) return fail(MB_ERR_OOM, "host allocation failed");
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    MB_CUDA(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
    MB_CUDA(cudaMalloc(&ctx->scratch, sizeof(double) * std::max(mb::sum_scratch_doubles(), mb::dot_scratch_doubles())));
    MB_CUDA(cudaMallocHost(&ctx->host_scalar, sizeof(double)));
    MB_CUDA(cudaEventCreate(&ctx->ev0));
    MB_CUDA(cudaEventCreate(&ctx->ev1));
    *out = ctx;
    return MB_OK;
}

int32_t mb_shutdown(mb_ctx* ctx) {
    if (!ctx) return MB_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->scratch) cudaFree(ctx->scratch);
    if (ctx->vec_ws) cudaFree(ctx->vec_ws);
    if (ctx->int_ws) cudaFree(ctx->int_ws);
    if (ctx->int_host) cudaFreeHost(ctx->int_host);
    if (ctx->host_scalar) cudaFreeHost(ctx->host_scalar);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->h2d_stream) cudaStreamDestroy(ctx->h2d_stream);
    if (ctx->d2h_stream) cudaStreamDestroy(ctx->d2h_stream);
    if (ctx->workspace) cudaFree(ctx->workspace);
    if (ctx->ozaki_ws) cudaFree(ctx->ozaki_ws);
    delete ctx;
    return MB_OK;
}

int32_t mb_set_stream(mb_ctx* ctx, void* cuda_stream) {
    if (!ctx) return fail(MB_ERR_INVALID_ARG, "null context");
    ctx->stream = static_cast<cudaStream_t>(cuda_stream);
    return MB_OK;
}

int32_t mb_reset_stream(mb_ctx* ctx) {
    if (!ctx) return fail(MB_ERR_INVALID_ARG, "null context");
    ctx->stream = ctx->own_stream;
    return MB_OK;
}

int32_t mb_synchronize(mb_ctx* ctx) {
    MB_CTX(ctx);
    MB_CUDA(cudaStreamSynchronize(ctx->stream));
    return MB_OK;
}

int64_t mb_launch_count(mb_ctx* ctx) { return ctx ? (int64_t)ctx->launches.load() : 0; }

int32_t mb_timer_start(mb_ctx* ctx) {
    MB_CTX(ctx);
    MB_LOCK(ctx);
    MB_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
    return MB_OK;
}
int32_t mb_timer_stop(mb_ctx* ctx, float* ms_out) {
    MB_CTX(ctx);
    MB_LOCK(ctx);
    if (!ms_out) return fail(MB_ERR_INVALID_ARG, "null ms_out");
    MB_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    MB_CUDA(cudaEventSynchronize(ctx->ev1));
    MB_CUDA(cudaEventElapsedTime(ms_out, ctx->ev0, ctx->ev1));
    return MB_OK;
}

// ---------------------------------------------------------------------------------- blocks
int32_t mb_block_alloc(mb_ctx* ctx, int32_t rows, int32_t cols, mb_dtype dtype, mb_block** out) {
    MB_CTX(ctx);
    if (!out || rows < 0 || cols < 0 || dtype < 0 || dtype > 2) return fail(MB_ERR_INVALID_ARG, "mb_block_alloc: bad argument");
    int32_t r = new_block(out);
    if (r) return r;
    mb_block* b = *out;
    b->rows = rows; b->cols = cols; b->ld = rows > 0 ? rows : 1; b->dtype = dtype; b->owns = 1; b->device = ctx->device;
    const size_t bytes = (size_t)rows * (size_t)cols * elem_size(dtype);
    if (bytes) {
        cudaError_t e = cudaMalloc(&b->data, bytes);
        if (e != cudaSuccess) { delete b; *out = nullptr; return cuda_fail(e, "cudaMalloc(block)"); }
    }
    return MB_OK;
}

int32_t mb_block_wrap(mb_ctx* ctx, void* device_ptr, int64_t offset, int32_t rows, int32_t cols, int32_t ld,
                      int32_t is_transpose, mb_dtype dtype, mb_block** out) {
    if (!ctx) return fail(MB_ERR_INVALID_ARG, "null context");
    if (!out || rows < 0 || cols < 0 || offset < 0 || dtype < 0 || dtype > 2)
        return fail(MB_ERR_INVALID_ARG, "mb_block_wrap: bad argument");
    const int minor = is_transpose ? cols : rows;
    if (ld < (minor > 0 ? minor : 1)) return fail(MB_ERR_INVALID_ARG, "mb_block_wrap: ld %d < %d", ld, minor);
    int32_t r = new_block(out);
    if (r) return r;
    mb_block* b = *out;
    b->data = device_ptr; b->offset = offset; b->rows = rows; b->cols = cols; b->ld = ld;
    b->is_transpose = is_transpose ? 1 : 0; b->dtype = dtype; b->owns = 0; b->device = ctx->device;
    return MB_OK;
}

int32_t mb_block_free(mb_ctx* ctx, mb_block* blk) {
    if (!blk) return MB_OK;
    if (blk->owns && blk->data) {
        if (ctx) cudaSetDevice(ctx->device);
        cudaFree(blk->data);
    }
    delete blk;
    return MB_OK;
}

int32_t mb_block_info(const mb_block* blk, int32_t* rows, int32_t* cols, int32_t* ld, int32_t* is_transpose,
                      int32_t* dtype, void** device_ptr) {
    if (!blk) return fail(MB_ERR_INVALID_ARG, "null block");
    if (rows) *rows = blk->rows;
    if (cols) *cols = blk->cols;
    if (ld) *ld = blk->ld;
    if (is_transpose) *is_transpose = blk->is_transpose;
    if (dtype) *dtype = blk->dtype;
    if (device_ptr) *device_ptr = elem_ptr(blk);
    return MB_OK;
}

int32_t mb_block_set_ready_event(mb_block* blk, void* cuda_event) {
    if (!blk) return fail(MB_ERR_INVALID_ARG, "null block");
    blk->ready_event = cuda_event;
    return MB_OK;
}

int32_t mb_block_view_t(mb_ctx* ctx, const mb_block* blk, mb_block** out) {
    if (!ctx || !blk || !out) return fail(MB_ERR_INVALID_ARG, "mb_block_view_t: null argument");
    int32_t r = new_block(out);
    if (r) return r;
    **out = *blk;
    (*out)->owns = 0;
    std::swap((*out)->rows, (*out)->cols);
    (*out)->is_transpose = !blk->is_transpose;
    return MB_OK;
}

int32_t mb_block_slice(mb_ctx* ctx, const mb_block* blk, int32_t r0, int32_t r1, int32_t c0, int32_t c1, mb_block** out) {
    if (!ctx || !blk || !out) return fail(MB_ERR_INVALID_ARG, "mb_block_slice: null argument");
    if (r0 < 0 || r1 < r0 || r1 > blk->rows || c0 < 0 || c1 < c0 || c1 > blk->cols)
        return fail(MB_ERR_INVALID_ARG, "mb_block_slice: range [%d,%d)x[%d,%d) outside %dx%d", r0, r1, c0, c1, blk->rows, blk->cols);
    int32_t r = new_block(out);
    if (r) return r;
    **out = *blk;
    (*out)->owns = 0;
    (*out)->rows = r1 - r0;
    (*out)->cols = c1 - c0;
    (*out)->offset = blk->offset + r0 * rs(blk) + c0 * cs(blk);
    return MB_OK;
}

int32_t mb_block_upload(mb_ctx* ctx, const double* host, int64_t offset, int32_t rows, int32_t cols, int32_t ld,
                        int32_t is_transpose, mb_dtype store_as, mb_block** out) {
    MB_CTX(ctx);
    if (!host || !out || rows < 0 || cols < 0 || offset < 0) return fail(MB_ERR_INVALID_ARG, "mb_block_upload: bad argument");
    const int minor = is_transpose ? cols : rows, major = is_transpose ? rows : cols;
    if (ld < (minor > 0 ? minor : 1)) return fail(MB_ERR_INVALID_ARG, "mb_block_upload: ld %d < %d", ld, minor);
    int32_t r = mb_block_alloc(ctx, rows, cols, store_as, out);
    if (r) return r;
    if (rows == 0 || cols == 0) return MB_OK;
    // stage the raw (minor x major) host array, then one device kernel packs / transposes / rounds it
    mb_block* dst = *out;
    const bool direct = (store_as == MB_F64) && !is_transpose;
    if (direct) {
        cudaError_t e = cudaMemcpy2DAsync(dst->data, (size_t)rows * 8, host + offset, (size_t)ld * 8, (size_t)rows * 8,
                                          (size_t)cols, cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) { mb_block_free(ctx, dst); *out = nullptr; return cuda_fail(e, "cudaMemcpy2DAsync(H2D)"); }
        MB_CUDA(cudaStreamSynchronize(ctx->stream));
        return MB_OK;
    }
    double* stage = nullptr;
    MB_CUDA(cudaMalloc(&stage, (size_t)minor * major * 8));
    cudaError_t e = cudaMemcpy2DAsync(stage, (size_t)minor * 8, host + offset, (size_t)ld * 8, (size_t)minor * 8,
                                      (size_t)major, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) { cudaFree(stage); mb_block_free(ctx, dst); *out = nullptr; return cuda_fail(e, "cudaMemcpy2DAsync(H2D)"); }
    mb_block src;
    src.data = stage; src.rows = rows; src.cols = cols; src.ld = minor; src.is_transpose = is_transpose ? 1 : 0; src.dtype = MB_F64;
    r = copy_convert(ctx, &src, dst);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(stage);
    if (r) { mb_block_free(ctx, dst); *out = nullptr; }
    return r;
}

int32_t mb_block_download(mb_ctx* ctx, const mb_block* blk, double* host, int32_t ld) {
    MB_CTX(ctx);
    if (!blk || !host) return fail(MB_ERR_INVALID_ARG, "mb_block_download: null argument");
    if (ld < blk->rows) return fail(MB_ERR_INVALID_ARG, "mb_block_download: ld %d < rows %d", ld, blk->rows);
    if (blk->rows == 0 || blk->cols == 0) return MB_OK;
    const double* src = nullptr;
    size_t src_pitch = 0;
    double* stage = nullptr;
    if (blk->dtype == MB_F64 && !blk->is_transpose) {
        src = f64_ptr(blk);
        src_pitch = (size_t)blk->ld * 8;
    } else {
        MB_CUDA(cudaMalloc(&stage, (size_t)blk->rows * blk->cols * 8));
        mb_block tmp;
        tmp.data = stage; tmp.rows = blk->rows; tmp.cols = blk->cols; tmp.ld = blk->rows; tmp.dtype = MB_F64;
        int32_t r = copy_convert(ctx, blk, &tmp);
        if (r) { cudaFree(stage); return r; }
        src = stage;
        src_pitch = (size_t)blk->rows * 8;
    }
    cudaError_t e = cudaMemcpy2DAsync(host, (size_t)ld * 8, src, src_pitch, (size_t)blk->rows * 8, (size_t)blk->cols,
                                      cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (stage) cudaFree(stage);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpy2DAsync(D2H)");
    return MB_OK;
}

// ------------------------------------------------------------------------------------ GEMM
static int32_t dgemm_device_impl(mb_ctx* ctx, char transa, char transb, int32_t m, int32_t n, int32_t k, double alpha,
                                 const double* A, int32_t lda, const double* B, int32_t ldb, double beta, double* C,
                                 int32_t ldc, bool force_generic) {
    MB_CTX(ctx);
    MB_LOCK(ctx);
    const bool ta = (transa == 'T' || transa == 't' || transa == 'C' || transa == 'c');
    const bool tb = (transb == 'T' || transb == 't' || transb == 'C' || transb == 'c');
    if (!ta && !(transa == 'N' || transa == 'n')) return fail(MB_ERR_INVALID_ARG, "dgemm: transa '%c'", transa);
    if (!tb && !(transb == 'N' || transb == 'n')) return fail(MB_ERR_INVALID_ARG, "dgemm: transb '%c'", transb);
    if (m < 0 || n < 0 || k < 0) return fail(MB_ERR_INVALID_ARG, "dgemm: negative dimension");
    const int nrowa = ta ? k : m, nrowb = tb ? n : k;
    if (lda < (nrowa > 1 ? nrowa : 1) || ldb < (nrowb > 1 ? nrowb : 1) || ldc < (m > 1 ? m : 1))
        return fail(MB_ERR_INVALID_ARG, "dgemm: leading dimension too small (lda=%d ldb=%d ldc=%d)", lda, ldb, ldc);
    if (m == 0 || n == 0) return MB_OK;
    if (!C || (k > 0 && alpha != 0.0 && (!A || !B))) return fail(MB_ERR_INVALID_ARG, "dgemm: null pointer");
    int launches = 0;
    if (ctx->fp64_mode != MB_FP64_NATIVE && !force_generic && !ta && !tb && alpha == 1.0 && (beta == 0.0 || beta == 1.0) &&
        m >= 256 && n >= 256 && k >= 256 && mb::ozaki_supported(m, n, k, ctx->fp64_slices, ctx->fp64_bits)) {
        const size_t need = mb::ozaki_workspace_bytes(m, n, k, ctx->fp64_slices);
        if (need > ctx->ozaki_ws_bytes) {
            if (ctx->ozaki_ws) { MB_CUDA(cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->ozaki_ws); ctx->ozaki_ws = nullptr; ctx->ozaki_ws_bytes = 0; }
            MB_CUDA(cudaMalloc(&ctx->ozaki_ws, need));
            ctx->ozaki_ws_bytes = need;
        }
        cudaError_t e = mb::gemm_f64_ozaki(m, n, k, A, lda, B, ldb, C, ldc, beta == 1.0, ctx->fp64_slices, ctx->fp64_bits, ctx->ozaki_ws,
                                           ctx->num_sms, ctx->stream, &launches);
        if (e == cudaSuccess) { ctx->launches += launches; return MB_OK; }
        if (e != cudaErrorNotSupported) return cuda_fail(e, "gemm_f64_ozaki");
        cudaGetLastError();
        launches = 0;
    }
    MB_CUDA(mb::gemm_f64(ta, tb, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, ctx->num_sms, ctx->stream, force_generic, &launches));
    ctx->launches += launches;
    return MB_OK;
}

int32_t mb_set_fp64_mode(mb_ctx* ctx, int32_t mode, int32_t slices) {
    if (!ctx) return fail(MB_ERR_INVALID_ARG, "null context");
    if (mode != MB_FP64_NATIVE && mode != MB_FP64_INT8_SPLIT && mode != MB_FP64_INT8_SPLIT8)
        return fail(MB_ERR_INVALID_ARG, "mb_set_fp64_mode: unknown mode %d", mode);
    if (mode != MB_FP64_NATIVE && (slices < 2 || slices > 8)) return fail(MB_ERR_INVALID_ARG, "mb_set_fp64_mode: slices must be in 2..8");
    ctx->fp64_mode = mode;
    if (mode != MB_FP64_NATIVE) { ctx->fp64_slices = slices; ctx->fp64_bits = (mode == MB_FP64_INT8_SPLIT8) ? 8 : 7; }
    return MB_OK;
}

int32_t mb_dgemm_device(mb_ctx* ctx, char transa, char transb, int32_t m, int32_t n, int32_t k, double alpha,
                        const double* A, int32_t lda, const double* B, int32_t ldb, double beta, double* C, int32_t ldc) {
    return dgemm_device_impl(ctx, transa, transb, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, false);
}
int32_t mb_dgemm_device_generic(mb_ctx* ctx, char transa, char transb, int32_t m, int32_t n, int32_t k, double alpha,
                                const double* A, int32_t lda, const double* B, int32_t ldb, double beta, double* C,
                                int32_t ldc) {
    return dgemm_device_impl(ctx, transa, transb, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, true);
}

int32_t mb_dgemm_host(mb_ctx* ctx, char transa, char transb, int32_t m, int32_t n, int32_t k, double alpha,
                      const double* a, int64_t a_offset, int32_t lda, const double* b, int64_t b_offset, int32_t ldb,
                      double beta, double* c, int64_t c_offset, int32_t ldc) {
    MB_CTX(ctx);
    const bool ta = (transa == 'T' || transa == 't'), tb = (transb == 'T' || transb == 't');
    if (m < 0 || n < 0 || k < 0) return fail(MB_ERR_INVALID_ARG, "dgemm: negative dimension");
    if (m == 0 || n == 0) return MB_OK;
    if (!a || !b || !c) return fail(MB_ERR_INVALID_ARG, "dgemm: null host array");
    const int ra = ta ? k : m, ca = ta ? m : k, rb = tb ? n : k, cb = tb ? k : n;
    if (lda < (ra > 1 ? ra : 1) || ldb < (rb > 1 ? rb : 1) || ldc < (m > 1 ? m : 1))
        return fail(MB_ERR_INVALID_ARG, "dgemm: leading dimension too small");
    // device staging is packed with an even leading dimension so the TMA path is always eligible
    auto even = [](int x) { return (x + 1) & ~1; };
    const int dlda = even(ra > 0 ? ra : 1), dldb = even(rb > 0 ? rb : 1), dldc = even(m);
    double *dA = nullptr, *dB = nullptr, *dC = nullptr;
    cudaError_t e = cudaSuccess;
    auto cleanup = [&]() { if (dA) cudaFree(dA); if (dB) cudaFree(dB); if (dC) cudaFree(dC); };
    if (k > 0) {
        if ((e = cudaMalloc(&dA, (size_t)dlda * ca * 8)) != cudaSuccess) { cleanup(); return cuda_fail(e, "cudaMalloc(A)"); }
        if ((e = cudaMalloc(&dB, (size_t)dldb * cb * 8)) != cudaSuccess) { cleanup(); return cuda_fail(e, "cudaMalloc(B)"); }
    }
    if ((e = cudaMalloc(&dC, (size_t)dldc * n * 8)) != cudaSuccess) { cleanup(); return cuda_fail(e, "cudaMalloc(C)"); }
    if (k > 0) {
        e = cudaMemcpy2DAsync(dA, (size_t)dlda * 8, a + a_offset, (size_t)lda * 8, (size_t)ra * 8, ca, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess)
            e = cudaMemcpy2DAsync(dB, (size_t)dldb * 8, b + b_offset, (size_t)ldb * 8, (size_t)rb * 8, cb, cudaMemcpyHostToDevice, ctx->stream);
    }
    if (e == cudaSuccess && beta != 0.0)
        e = cudaMemcpy2DAsync(dC, (size_t)dldc * 8, c + c_offset, (size_t)ldc * 8, (size_t)m * 8, n, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) { cleanup(); return cuda_fail(e, "H2D copy"); }
    int32_t r = dgemm_device_impl(ctx, transa, transb, m, n, k, alpha, dA, dlda, dB, dldb, beta, dC, dldc, false);
    if (r == MB_OK) {
        e = cudaMemcpy2DAsync(c + c_offset, (size_t)ldc * 8, dC, (size_t)dldc * 8, (size_t)m * 8, n, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) r = cuda_fail(e, "D2H copy");
    }
    cleanup();
    return r;
}

int32_t mb_block_gemm(mb_ctx* ctx, const mb_block* A, const mb_block* B, mb_block* C, int32_t accumulate) {
    MB_CTX(ctx);
    if (!A || !B || !C) return fail(MB_ERR_INVALID_ARG, "mb_block_gemm: null block");
    if (A->cols != B->rows)
        return fail(MB_ERR_DIM_MISMATCH, "Dimension mismatch during matrix-matrix multiplication: %d vs %d", A->cols, B->rows);
    if (C->rows != A->rows || C->cols != B->cols)
        return fail(MB_ERR_DIM_MISMATCH, "mb_block_gemm: result block is %dx%d, expected %dx%d", C->rows, C->cols, A->rows, B->cols);
    const int M = A->rows, N = B->cols, K = A->cols;
    if (A->dtype == MB_F64 && B->dtype == MB_F64 && C->dtype == MB_F64) {
        // degenerate shapes are HBM-bound vector kernels, not tensor-core tiles
        if (N == 1 && M > 1) return mb_block_gemv(ctx, A, B, C, accumulate);                 // matrix x column
        if (M == 1 && N > 1) {                                                              // row x matrix = (B^T a^T)^T
            mb_block bt = *B;
            bt.is_transpose = !B->is_transpose;
            std::swap(bt.rows, bt.cols);
            bt.owns = 0;
            return mb_block_gemv(ctx, &bt, A, C, accumulate);
        }
        if (K == 1 && !accumulate && M > 1 && N > 1) return mb_block_ger(ctx, A, B, C);     // column x row
        if (!C->is_transpose) {
            return dgemm_device_impl(ctx, A->is_transpose ? 'T' : 'N', B->is_transpose ? 'T' : 'N', M, N, K, 1.0, f64_ptr(A),
                                     A->ld, f64_ptr(B), B->ld, accumulate ? 1.0 : 0.0, f64_ptr(C), C->ld, false);
        }
        // row-major result (DenseVecMatrix rows, matrix/DenseVecMatrix.scala:1660-1680): C^T = B^T * A^T,
        // where X^T of a transposed view is the plain column-major array underneath.
        return dgemm_device_impl(ctx, B->is_transpose ? 'N' : 'T', A->is_transpose ? 'N' : 'T', N, M, K, 1.0, f64_ptr(B),
                                 B->ld, f64_ptr(A), A->ld, accumulate ? 1.0 : 0.0, f64_ptr(C), C->ld, false);
    }
    if (A->dtype == MB_BF16 && B->dtype == MB_BF16 && (C->dtype == MB_F32 || C->dtype == MB_BF16)) {
        int launches = 0;
        cudaError_t e;
        if (!C->is_transpose) {
            e = mb::gemm_bf16(A->is_transpose, B->is_transpose, M, N, K, elem_ptr(A), A->ld, elem_ptr(B), B->ld,
                              elem_ptr(C), C->ld, C->dtype == MB_F32, accumulate != 0, ctx->num_sms, ctx->stream, &launches);
        } else {
            e = mb::gemm_bf16(!B->is_transpose, !A->is_transpose, N, M, K, elem_ptr(B), B->ld, elem_ptr(A), A->ld,
                              elem_ptr(C), C->ld, C->dtype == MB_F32, accumulate != 0, ctx->num_sms, ctx->stream, &launches);
        }
        if (e == cudaErrorNotSupported)
            return fail(MB_ERR_UNSUPPORTED, "mb_block_gemm(bf16): operands must be 16-byte aligned with ld %% 8 == 0");
        if (e != cudaSuccess) return cuda_fail(e, "gemm_bf16");
        ctx->launches += launches;
        return MB_OK;
    }
    return fail(MB_ERR_UNSUPPORTED, "mb_block_gemm: unsupported dtype combination (%d,%d)->%d", A->dtype, B->dtype, C->dtype);
}

int32_t mb_matmul_blocked_subset(mb_ctx* ctx, mb_block* const* A_tiles, mb_block* const* B_tiles, int32_t m, int32_t k,
                                 int32_t n, mb_block* const* C_tiles, const int32_t* c_ids, int32_t num_c) {
    MB_CTX(ctx);
    if (!A_tiles || !B_tiles || !C_tiles || !c_ids || m <= 0 || k <= 0 || n <= 0 || num_c < 0)
        return fail(MB_ERR_INVALID_ARG, "mb_matmul_blocked: bad argument");
    for (int c = 0; c < num_c; ++c) {
        const int id = c_ids[c];
        if (id < 0 || id >= m * n || !C_tiles[id]) return fail(MB_ERR_INVALID_ARG, "mb_matmul_blocked: bad C id %d", id);
        const int i = id / n, j = id % n;
        for (int kk = 0; kk < k; ++kk) {
            const mb_block *a = A_tiles[i * k + kk], *b = B_tiles[kk * n + j];
            if (!a || !b) return fail(MB_ERR_INVALID_ARG, "mb_matmul_blocked: missing tile for C(%d,%d), kk=%d", i, j, kk);
            if (a->cols != b->rows)
                return fail(MB_ERR_DIM_MISMATCH, "Dimension mismatch during matrix-matrix multiplication: %d vs %d", a->cols, b->rows);
            if (C_tiles[id]->rows != a->rows || C_tiles[id]->cols != b->cols)
                return fail(MB_ERR_DIM_MISMATCH, "mb_matmul_blocked: C(%d,%d) is %dx%d, expected %dx%d", i, j, C_tiles[id]->rows,
                            C_tiles[id]->cols, a->rows, b->cols);
        }
    }
    // ---- grouped single launch when every operand is an fp64 column-major ('N') block ----
    bool groupable = num_c > 0 && ctx->fp64_mode == MB_FP64_NATIVE;
    std::vector<const double*> Ap(m * k, nullptr), Bp(k * n, nullptr);
    std::vector<double*> Cp(m * n, nullptr);
    std::vector<long long> lda(m * k, 2), ldb(k * n, 2), ldc(m * n, 2);
    std::vector<int> row_len(m, -1), k_len(k, -1), col_len(n, -1);    // -1 = not seen yet
    for (int c = 0; c < num_c && groupable; ++c) {
        const int id = c_ids[c], i = id / n, j = id % n;
        const mb_block* cb = C_tiles[id];
        groupable = cb->dtype == MB_F64 && !cb->is_transpose;
        Cp[id] = f64_ptr(cb); ldc[id] = cb->ld;
        for (int kk = 0; kk < k && groupable; ++kk) {
            const mb_block *a = A_tiles[i * k + kk], *b = B_tiles[kk * n + j];
            groupable = a->dtype == MB_F64 && b->dtype == MB_F64 && !a->is_transpose && !b->is_transpose && a->rows > 0 &&
                        a->cols > 0 && b->cols > 0;
            Ap[i * k + kk] = f64_ptr(a); lda[i * k + kk] = a->ld;
            Bp[kk * n + j] = f64_ptr(b); ldb[kk * n + j] = b->ld;
            // the k-slab count is shared by all C blocks: every A(.,kk) must have the same column count
            if (k_len[kk] >= 0 && k_len[kk] != a->cols) groupable = false;
            if (row_len[i] >= 0 && row_len[i] != a->rows) groupable = false;
            if (col_len[j] >= 0 && col_len[j] != b->cols) groupable = false;
            k_len[kk] = a->cols;
            row_len[i] = a->rows; col_len[j] = b->cols;
        }
    }
    if (groupable) {
        int launches = 0;
        cudaError_t e = mb::gemm_f64_grouped(m, k, n, c_ids, num_c, Ap.data(), lda.data(), Bp.data(), ldb.data(), Cp.data(),
                                             ldc.data(), row_len.data(), k_len.data(), col_len.data(), ctx->num_sms, ctx->stream,
                                             &launches);
        if (e == cudaSuccess) { ctx->launches += launches; return MB_OK; }
        if (e != cudaErrorNotSupported) return cuda_fail(e, "gemm_f64_grouped");
        cudaGetLastError();
    }
    // ---- fallback: seq order of matrix/BlockMatrix.scala:163,168 (p = i*n*k + j*k + kk), the kk partials of C(i,j)
    //      (reduceByKey at :177) accumulated in place, kk ascending ----
    for (int c = 0; c < num_c; ++c) {
        const int id = c_ids[c], i = id / n, j = id % n;
        mb_block* cb = C_tiles[id];
        // bf16 tiles: fold the kk-sum into ONE tcgen05 launch per C block (K segments; accumulator stays in TMEM)
        bool seg_ok = k <= 8 && !cb->is_transpose && (cb->dtype == MB_F32 || cb->dtype == MB_BF16);
        const void* Ap[8]; const void* Bp[8]; long long la[8], lb[8]; int Ks[8];
        for (int kk = 0; kk < k && seg_ok; ++kk) {
            const mb_block *a = A_tiles[i * k + kk], *b = B_tiles[kk * n + j];
            seg_ok = a->dtype == MB_BF16 && b->dtype == MB_BF16 && !a->is_transpose && !b->is_transpose && a->cols > 0;
            Ap[kk] = elem_ptr(a); Bp[kk] = elem_ptr(b); la[kk] = a->ld; lb[kk] = b->ld; Ks[kk] = a->cols;
        }
        if (seg_ok) {
            // The tensor cores add into the fp32 TMEM accumulator with truncation, so one accumulation chain drifts by about
            // (chain length in K) * 5e-9 relative on same-sign data (measured: 3.5e-4 at K = 65536).  Chains are therefore
            // capped (MARLIN_B200_BF16_KCHAIN, default 8192; 0 = unlimited): an fp32 C block is produced by several
            // launches whose epilogues add into C with round-to-nearest.  bf16 C blocks keep the single launch (one rounding).
            static const long long kchain = [] { const char* e = getenv("MARLIN_B200_BF16_KCHAIN"); return e ? atoll(e) : 8192ll; }();
            long long total_k = 0;
            for (int kk = 0; kk < k; ++kk) total_k += Ks[kk];
            int launches = 0;
            cudaError_t e = cudaSuccess;
            if (cb->dtype != MB_F32 || kchain <= 0 || total_k <= kchain) {
                e = mb::gemm_bf16_segments(false, false, cb->rows, cb->cols, k, Ks, Ap, la, Bp, lb, elem_ptr(cb), cb->ld,
                                           cb->dtype == MB_F32, false, ctx->num_sms, ctx->stream, &launches);
            } else {
                const void* sa[8]; const void* sb[8]; long long sla[8], slb[8]; int sk[8];
                int ns = 0, group = 0;
                long long in_group = 0;
                auto flush = [&]() {
                    if (ns == 0 || e != cudaSuccess) return;
                    e = mb::gemm_bf16_segments(false, false, cb->rows, cb->cols, ns, sk, sa, sla, sb, slb, elem_ptr(cb), cb->ld, true,
                                               group > 0, ctx->num_sms, ctx->stream, &launches);
                    ++group; ns = 0; in_group = 0;
                };
                for (int kk = 0; kk < k && e == cudaSuccess; ++kk)
                    for (int k0 = 0; k0 < Ks[kk] && e == cudaSuccess;) {
                        const int len = (int)std::min<long long>(Ks[kk] - k0, kchain - in_group);
                        sa[ns] = static_cast<const char*>(Ap[kk]) + (size_t)k0 * la[kk] * 2;       // columns k0.. of A(i,kk)
                        sb[ns] = static_cast<const char*>(Bp[kk]) + (size_t)k0 * 2;                // rows k0.. of B(kk,j)
                        sla[ns] = la[kk]; slb[ns] = lb[kk]; sk[ns] = len;
                        ++ns; in_group += len; k0 += len;
                        if (in_group >= kchain || ns == 8) flush();
                    }
                flush();
            }
            if (e == cudaSuccess) { ctx->launches += launches; continue; }
            if (e != cudaErrorNotSupported) return cuda_fail(e, "gemm_bf16_segments");
            cudaGetLastError();
        }
        for (int kk = 0; kk < k; ++kk) {
            int32_t r = mb_block_gemm(ctx, A_tiles[i * k + kk], B_tiles[kk * n + j], C_tiles[id], kk > 0);
            if (r) return r;
        }
    }
    return MB_OK;
}

int32_t mb_matmul_blocked(mb_ctx* ctx, mb_block* const* A_tiles, mb_block* const* B_tiles, int32_t m, int32_t k,
                          int32_t n, mb_block* const* C_tiles) {
    if (m <= 0 || k <= 0 || n <= 0) return fail(MB_ERR_INVALID_ARG, "mb_matmul_blocked: bad argument");
    std::vector<int32_t> ids(m * n);
    for (int c = 0; c < m * n; ++c) ids[c] = c;
    return mb_matmul_blocked_subset(ctx, A_tiles, B_tiles, m, k, n, C_tiles, ids.data(), m * n);
}

int32_t mb_matmul_blocked_host(mb_ctx* ctx, const double* const* A_host, const double* const* B_host, int32_t m,
                               int32_t k, int32_t n, const int32_t* row_len, const int32_t* k_len, const int32_t* col_len,
                               double* const* C_host) {
    MB_CTX(ctx);
    MB_LOCK(ctx);
    if (!A_host || !B_host || !C_host || !row_len || !k_len || !col_len || m <= 0 || k <= 0 || n <= 0)
        return fail(MB_ERR_INVALID_ARG, "mb_matmul_blocked_host: bad argument");
    if (!ctx->h2d_stream) {
        MB_CUDA(cudaStreamCreateWithFlags(&ctx->h2d_stream, cudaStreamNonBlocking));
        MB_CUDA(cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking));
    }
    // device layout: every tile gets an even leading dimension and a 256-byte aligned slot (TMA eligibility)
    auto even = [](int x) { return (x + 1) & ~1; };
    auto slot = [](size_t bytes) { return (bytes + 255) & ~size_t(255); };
    std::vector<size_t> offA(m * k), offB(k * n), offC(m * n);
    size_t total = 0;
    for (int i = 0; i < m; ++i)
        for (int kk = 0; kk < k; ++kk) { offA[i * k + kk] = total; total += slot((size_t)even(row_len[i]) * k_len[kk] * 8); }
    for (int kk = 0; kk < k; ++kk)
        for (int j = 0; j < n; ++j) { offB[kk * n + j] = total; total += slot((size_t)even(k_len[kk]) * col_len[j] * 8); }
    for (int i = 0; i < m; ++i)
        for (int j = 0; j < n; ++j) { offC[i * n + j] = total; total += slot((size_t)even(row_len[i]) * col_len[j] * 8); }
    if (total > ctx->workspace_bytes) {
        if (ctx->workspace) { MB_CUDA(cudaDeviceSynchronize()); cudaFree(ctx->workspace); ctx->workspace = nullptr; ctx->workspace_bytes = 0; }
        MB_CUDA(cudaMalloc(&ctx->workspace, total));
        ctx->workspace_bytes = total;
    }
    char* base = static_cast<char*>(ctx->workspace);
    std::vector<cudaEvent_t> evA(m * k, nullptr), evB(k * n, nullptr), evC(m * n, nullptr);
    cudaEvent_t ev_start = nullptr, ev_done = nullptr;
    int32_t rc = MB_OK;
    cudaError_t e = cudaSuccess;
    auto upload = [&](bool isA, int idx, int rows, int cols, const double* host, size_t off, cudaEvent_t& ev) {
        if (ev || e != cudaSuccess) return;
        e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
        if (e != cudaSuccess) return;
        if (rows > 0 && cols > 0)
            e = cudaMemcpy2DAsync(base + off, (size_t)even(rows) * 8, host, (size_t)rows * 8, (size_t)rows * 8, cols,
                                  cudaMemcpyHostToDevice, ctx->h2d_stream);
        if (e == cudaSuccess) e = cudaEventRecord(ev, ctx->h2d_stream);
        (void)isA; (void)idx;
    };
    // the workspace may still be read by a previous call on ctx->stream / d2h_stream: order behind them
    e = cudaEventCreateWithFlags(&ev_start, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventRecord(ev_start, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->h2d_stream, ev_start, 0);
    // one block product restricted to columns [c0, c1) of B(kk,j) / C(i,j)
    auto gemm_cols = [&](int i, int j, int kk, int c0, int c1) {
        const int lda8 = even(row_len[i]) > 0 ? even(row_len[i]) : 1, ldb8 = even(k_len[kk]) > 0 ? even(k_len[kk]) : 1;
        rc = dgemm_device_impl(ctx, 'N', 'N', row_len[i], c1 - c0, k_len[kk], 1.0, reinterpret_cast<double*>(base + offA[i * k + kk]), lda8,
                               reinterpret_cast<double*>(base + offB[kk * n + j]) + (size_t)c0 * ldb8, ldb8, kk > 0 ? 1.0 : 0.0,
                               reinterpret_cast<double*>(base + offC[i * n + j]) + (size_t)c0 * lda8, lda8, false);
    };
    std::vector<cudaEvent_t> chunk_events;
    for (int i = 0; i < m && e == cudaSuccess && rc == MB_OK; ++i)
        for (int j = 0; j < n && e == cudaSuccess && rc == MB_OK; ++j) {
            for (int kk = 0; kk < k && e == cudaSuccess && rc == MB_OK; ++kk) {
                const bool first_product = (i == 0 && j == 0 && kk == 0);
                const bool last_product = (i == m - 1 && j == n - 1 && kk == k - 1);
                if (first_product && !last_product && k_len[kk] >= 1024 && row_len[i] > 0 && col_len[j] > 0) {
                    // The first product is split along K: the GEMM on chunk q needs only columns [k0,k1) of A and rows
                    // [k0,k1) of B, so the tensor cores start after a quarter of each tile has crossed PCIe and the rest
                    // of both uploads hides behind the partial products (accumulated in place, beta = 1).
                    const int nk = 4;
                    const int lda8 = even(row_len[i]), ldb8 = even(k_len[kk]);
                    for (int q = 0; q < nk && e == cudaSuccess && rc == MB_OK; ++q) {
                        const int k0 = q == 0 ? 0 : (int)(((long long)k_len[kk] * q / nk) & ~15ll);
                        const int k1 = q == nk - 1 ? k_len[kk] : (int)(((long long)k_len[kk] * (q + 1) / nk) & ~15ll);
                        cudaEvent_t ev = nullptr;
                        e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
                        if (e != cudaSuccess) break;
                        chunk_events.push_back(ev);
                        e = cudaMemcpy2DAsync(base + offA[i * k + kk] + (size_t)k0 * lda8 * 8, (size_t)lda8 * 8,
                                              A_host[i * k + kk] + (size_t)k0 * row_len[i], (size_t)row_len[i] * 8,
                                              (size_t)row_len[i] * 8, k1 - k0, cudaMemcpyHostToDevice, ctx->h2d_stream);
                        if (e == cudaSuccess)
                            e = cudaMemcpy2DAsync(base + offB[kk * n + j] + (size_t)k0 * 8, (size_t)ldb8 * 8, B_host[kk * n + j] + k0,
                                                  (size_t)k_len[kk] * 8, (size_t)(k1 - k0) * 8, col_len[j], cudaMemcpyHostToDevice,
                                                  ctx->h2d_stream);
                        if (e == cudaSuccess) e = cudaEventRecord(ev, ctx->h2d_stream);
                        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ev, 0);
                        if (e != cudaSuccess) break;
                        rc = dgemm_device_impl(ctx, 'N', 'N', row_len[i], col_len[j], k1 - k0, 1.0,
                                               reinterpret_cast<double*>(base + offA[i * k + kk]) + (size_t)k0 * lda8, lda8,
                                               reinterpret_cast<double*>(base + offB[kk * n + j]) + k0, ldb8, (kk > 0 || q > 0) ? 1.0 : 0.0,
                                               reinterpret_cast<double*>(base + offC[i * n + j]), lda8, false);
                    }
                    if (e != cudaSuccess || rc != MB_OK) break;
                    // later users of these two tiles wait for the whole of them
                    e = cudaEventCreateWithFlags(&evA[i * k + kk], cudaEventDisableTiming);
                    if (e == cudaSuccess) e = cudaEventRecord(evA[i * k + kk], ctx->h2d_stream);
                    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&evB[kk * n + j], cudaEventDisableTiming);
                    if (e == cudaSuccess) e = cudaEventRecord(evB[kk * n + j], ctx->h2d_stream);
                    continue;
                }
                const int nch = ((first_product || last_product) && col_len[j] >= 1024) ? 4 : 1;
                // uploads in first-use order (seq = i*n*k + j*k + kk)
                upload(true, i * k + kk, row_len[i], k_len[kk], A_host[i * k + kk], offA[i * k + kk], evA[i * k + kk]);
                if (e != cudaSuccess) break;
                e = cudaStreamWaitEvent(ctx->stream, evA[i * k + kk], 0);
                if (e != cudaSuccess) break;
                if (nch == 1) {
                    upload(false, kk * n + j, k_len[kk], col_len[j], B_host[kk * n + j], offB[kk * n + j], evB[kk * n + j]);
                    if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, evB[kk * n + j], 0);
                    if (e != cudaSuccess) break;
                    gemm_cols(i, j, kk, 0, col_len[j]);
                    continue;
                }
                // The first product starts after A + a quarter of B has landed (B uploaded and multiplied in column
                // chunks); the last product hands each finished column chunk of C to the D2H stream at once.
                const bool b_pending = (evB[kk * n + j] == nullptr);
                const int ldb8 = even(k_len[kk]), ldc8 = even(row_len[i]);
                for (int q = 0; q < nch && e == cudaSuccess && rc == MB_OK; ++q) {
                    const int c0 = (int)((long long)col_len[j] * q / nch), c1 = (int)((long long)col_len[j] * (q + 1) / nch);
                    if (b_pending) {
                        cudaEvent_t ev = nullptr;
                        e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
                        if (e != cudaSuccess) break;
                        chunk_events.push_back(ev);
                        e = cudaMemcpy2DAsync(base + offB[kk * n + j] + (size_t)c0 * ldb8 * 8, (size_t)ldb8 * 8,
                                              B_host[kk * n + j] + (size_t)c0 * k_len[kk], (size_t)k_len[kk] * 8, (size_t)k_len[kk] * 8,
                                              c1 - c0, cudaMemcpyHostToDevice, ctx->h2d_stream);
                        if (e == cudaSuccess) e = cudaEventRecord(ev, ctx->h2d_stream);
                        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ev, 0);
                        if (e != cudaSuccess) break;
                        if (q == nch - 1) {          // later users of this B tile wait for the whole of it
                            e = cudaEventCreateWithFlags(&evB[kk * n + j], cudaEventDisableTiming);
                            if (e == cudaSuccess) e = cudaEventRecord(evB[kk * n + j], ctx->h2d_stream);
                        }
                    } else if (q == 0) {
                        e = cudaStreamWaitEvent(ctx->stream, evB[kk * n + j], 0);
                    }
                    if (e != cudaSuccess) break;
                    gemm_cols(i, j, kk, c0, c1);
                    if (rc != MB_OK) break;
                    if (last_product) {
                        cudaEvent_t ev = nullptr;
                        e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
                        if (e != cudaSuccess) break;
                        chunk_events.push_back(ev);
                        e = cudaEventRecord(ev, ctx->stream);
                        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->d2h_stream, ev, 0);
                        if (e == cudaSuccess && row_len[i] > 0 && c1 > c0)
                            e = cudaMemcpy2DAsync(C_host[i * n + j] + (size_t)c0 * row_len[i], (size_t)row_len[i] * 8,
                                                  base + offC[i * n + j] + (size_t)c0 * ldc8 * 8, (size_t)ldc8 * 8, (size_t)row_len[i] * 8,
                                                  c1 - c0, cudaMemcpyDeviceToHost, ctx->d2h_stream);
                    }
                }
            }
            if (e != cudaSuccess || rc != MB_OK) break;
            const bool chunked_out = (i == m - 1 && j == n - 1 && col_len[j] >= 1024);
            if (chunked_out) continue;               // already downloaded chunk by chunk
            e = cudaEventCreateWithFlags(&evC[i * n + j], cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventRecord(evC[i * n + j], ctx->stream);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->d2h_stream, evC[i * n + j], 0);
            if (e == cudaSuccess && row_len[i] > 0 && col_len[j] > 0)
                e = cudaMemcpy2DAsync(C_host[i * n + j], (size_t)row_len[i] * 8, base + offC[i * n + j], (size_t)even(row_len[i]) * 8,
                                      (size_t)row_len[i] * 8, col_len[j], cudaMemcpyDeviceToHost, ctx->d2h_stream);
        }
    if (e == cudaSuccess && rc == MB_OK) {
        // the call returns when every C tile is on the host; ctx->stream is ordered behind the downloads too
        e = cudaEventCreateWithFlags(&ev_done, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventRecord(ev_done, ctx->d2h_stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ev_done, 0);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->d2h_stream);
    } else {
        cudaStreamSynchronize(ctx->h2d_stream); cudaStreamSynchronize(ctx->stream); cudaStreamSynchronize(ctx->d2h_stream);
    }
    for (auto ev : evA) if (ev) cudaEventDestroy(ev);
    for (auto ev : evB) if (ev) cudaEventDestroy(ev);
    for (auto ev : evC) if (ev) cudaEventDestroy(ev);
    for (auto ev : chunk_events) if (ev) cudaEventDestroy(ev);
    if (ev_start) cudaEventDestroy(ev_start);
    if (ev_done) cudaEventDestroy(ev_done);
    if (rc != MB_OK) return rc;
    if (e != cudaSuccess) return cuda_fail(e, "mb_matmul_blocked_host");
    return MB_OK;
}

// DenseVecMatrix.multiply(B: BDM) for one row shard (matrix/DenseVecMatrix.scala:1660-1680): C_rows = A_rows * B with
// A_rows / C_rows row-major shards (transposed views) and B the broadcast matrix.
int32_t mb_matmul_rowsharded(mb_ctx* ctx, const mb_block* A_rows, const mb_block* B, mb_block* C_rows) {
    MB_CTX(ctx);
    if (!A_rows || !B || !C_rows) return fail(MB_ERR_INVALID_ARG, "mb_matmul_rowsharded: null block");
    if (A_rows->cols != B->rows)
        return fail(MB_ERR_DIM_MISMATCH, "Dimension mismatch during matrix-matrix multiplication: %d vs %d", A_rows->cols, B->rows);
    return mb_block_gemm(ctx, A_rows, B, C_rows, 0);
}

// The same for JVM-held rows: A_host is the shard's rows back to back (row-major, each row k doubles — exactly the
// `Array[Double]` a partition's rows are packed into at :1672-1675), B_host the column-major k x n broadcast matrix,
// C_host receives the row-major rows x n result.  Row chunks are pipelined: H2D of chunk c+1, the DMMA product of chunk
// c (C^T = B^T * A^T on the row-major data, no transposition pass) and D2H of chunk c-1 run on three streams over a
// ring of three device slots.
int32_t mb_matmul_rowsharded_host(mb_ctx* ctx, const double* A_host, int64_t rows, int32_t k, const double* B_host,
                                  int32_t n, double* C_host) {
    MB_CTX(ctx);
    MB_LOCK(ctx);
    if (rows < 0 || k < 0 || n < 0 || (rows > 0 && ((k > 0 && !A_host) || (n > 0 && !C_host))) || (k > 0 && n > 0 && !B_host))
        return fail(MB_ERR_INVALID_ARG, "mb_matmul_rowsharded_host: bad argument");
    if (rows == 0 || n == 0) return MB_OK;
    if (!ctx->h2d_stream) {
        MB_CUDA(cudaStreamCreateWithFlags(&ctx->h2d_stream, cudaStreamNonBlocking));
        MB_CUDA(cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking));
    }
    constexpr int SLOTS = 3;
    // ~256 MiB of A (or C, whichever is wider) per chunk, a multiple of 128 rows (whole GEMM tiles), at least one tile;
    // MARLIN_B200_ROWSHARD_CHUNK_MIB overrides the size (the tests use it to run many chunks on small inputs)
    long long chunk_mib = 256;
    if (const char* ev = getenv("MARLIN_B200_ROWSHARD_CHUNK_MIB")) chunk_mib = std::max(1, atoi(ev));
    long long chunk = (chunk_mib << 20) / (8ll * std::max(std::max(k, n), 1));
    chunk = std::max(128ll, chunk / 128 * 128);
    chunk = std::min<long long>(chunk, (rows + 127) / 128 * 128);
    const int kk = std::max(k, 1);
    auto slot = [](size_t bytes) { return (bytes + 255) & ~size_t(255); };
    const size_t bytesB = slot((size_t)kk * n * 8), bytesA = slot((size_t)chunk * kk * 8), bytesC = slot((size_t)chunk * n * 8);
    const size_t total = bytesB + SLOTS * (bytesA + bytesC);
    if (total > ctx->workspace_bytes) {
        if (ctx->workspace) { MB_CUDA(cudaDeviceSynchronize()); cudaFree(ctx->workspace); ctx->workspace = nullptr; ctx->workspace_bytes = 0; }
        MB_CUDA(cudaMalloc(&ctx->workspace, total));
        ctx->workspace_bytes = total;
    }
    char* base = static_cast<char*>(ctx->workspace);
    double* dB = reinterpret_cast<double*>(base);
    auto dA = [&](int s_) { return reinterpret_cast<double*>(base + bytesB + (size_t)s_ * (bytesA + bytesC)); };
    auto dC = [&](int s_) { return reinterpret_cast<double*>(base + bytesB + (size_t)s_ * (bytesA + bytesC) + bytesA); };
    cudaEvent_t ev_start = nullptr, ev_b = nullptr, ev_up[SLOTS] = {}, ev_gemm[SLOTS] = {}, ev_down[SLOTS] = {};
    cudaError_t e = cudaSuccess;
    int32_t rc = MB_OK;
    auto mk = [&](cudaEvent_t& ev) { if (e == cudaSuccess && !ev) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming); };
    mk(ev_start); mk(ev_b);
    for (int s_ = 0; s_ < SLOTS; ++s_) { mk(ev_up[s_]); mk(ev_gemm[s_]); mk(ev_down[s_]); }
    // the workspace may still be in use by an earlier call on ctx->stream
    if (e == cudaSuccess) e = cudaEventRecord(ev_start, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->h2d_stream, ev_start, 0);
    if (e == cudaSuccess && k > 0) e = cudaMemcpyAsync(dB, B_host, (size_t)k * n * 8, cudaMemcpyHostToDevice, ctx->h2d_stream);
    if (e == cudaSuccess) e = cudaEventRecord(ev_b, ctx->h2d_stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ev_b, 0);
    const long long nchunks = (rows + chunk - 1) / chunk;
    for (long long c = 0; c < nchunks && e == cudaSuccess && rc == MB_OK; ++c) {
        const int s_ = (int)(c % SLOTS);
        const long long r0 = c * chunk;
        const int nr = (int)std::min<long long>(chunk, rows - r0);
        if (c >= SLOTS) {                       // the slot's previous tenant: its GEMM has read A, its download has read C
            e = cudaStreamWaitEvent(ctx->h2d_stream, ev_gemm[s_], 0);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ev_down[s_], 0);
            if (e != cudaSuccess) break;
        }
        if (k > 0) e = cudaMemcpyAsync(dA(s_), A_host + (size_t)r0 * k, (size_t)nr * k * 8, cudaMemcpyHostToDevice, ctx->h2d_stream);
        if (e == cudaSuccess) e = cudaEventRecord(ev_up[s_], ctx->h2d_stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ev_up[s_], 0);
        if (e != cudaSuccess) break;
        // row-major (nr x n) C chunk == column-major (n x nr) C^T = B^T (n x k) * A^T (k x nr, the row-major chunk itself)
        rc = dgemm_device_impl(ctx, 'T', 'N', n, nr, k, 1.0, dB, kk, dA(s_), kk, 0.0, dC(s_), n, false);
        if (rc != MB_OK) break;
        e = cudaEventRecord(ev_gemm[s_], ctx->stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->d2h_stream, ev_gemm[s_], 0);
        if (e == cudaSuccess) e = cudaMemcpyAsync(C_host + (size_t)r0 * n, dC(s_), (size_t)nr * n * 8, cudaMemcpyDeviceToHost, ctx->d2h_stream);
        if (e == cudaSuccess) e = cudaEventRecord(ev_down[s_], ctx->d2h_stream);
    }
    if (e == cudaSuccess && rc == MB_OK) {
        // returns when every row is on the host; ctx->stream is ordered behind the downloads too
        for (int s_ = 0; s_ < SLOTS && e == cudaSuccess; ++s_)
            if (s_ < nchunks) e = cudaStreamWaitEvent(ctx->stream, ev_down[s_], 0);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->d2h_stream);
    } else {
        cudaStreamSynchronize(ctx->h2d_stream); cudaStreamSynchronize(ctx->stream); cudaStreamSynchronize(ctx->d2h_stream);
    }
    if (ev_start) cudaEventDestroy(ev_start);
    if (ev_b) cudaEventDestroy(ev_b);
    for (int s_ = 0; s_ < SLOTS; ++s_) {
        if (ev_up[s_]) cudaEventDestroy(ev_up[s_]);
        if (ev_gemm[s_]) cudaEventDestroy(ev_gemm[s_]);
        if (ev_down[s_]) cudaEventDestroy(ev_down[s_]);
    }
    if (rc != MB_OK) return rc;
    if (e != cudaSuccess) return cuda_fail(e, "mb_matmul_rowsharded_host");
    return MB_OK;
}

// ----------------------------------------------------------------------------- peer memory
int32_t mb_ipc_export(mb_ctx* ctx, const void* device_ptr, uint8_t handle_out[64], int64_t* offset_out, int64_t* alloc_bytes_out) {
    MB_CTX(ctx);
    if (!device_ptr || !handle_out || !offset_out || !alloc_bytes_out) return fail(MB_ERR_INVALID_ARG, "mb_ipc_export: null argument");
    long long off = 0, bytes = 0;
    MB_CUDA(mb::ipc_export(device_ptr, handle_out, &off, &bytes));
    *offset_out = off; *alloc_bytes_out = bytes;
    return MB_OK;
}
int32_t mb_ipc_open(mb_ctx* ctx, const uint8_t handle[64], void** base_out) {
    MB_CTX(ctx);
    if (!handle || !base_out) return fail(MB_ERR_INVALID_ARG, "mb_ipc_open: null argument");
    MB_CUDA(mb::ipc_open(handle, base_out));
    return MB_OK;
}
int32_t mb_ipc_close_all(mb_ctx* ctx) {
    MB_CTX(ctx);
    MB_CUDA(cudaDeviceSynchronize());
    MB_CUDA(mb::ipc_close_all());
    return MB_OK;
}
int32_t mb_flags_alloc(mb_ctx* ctx, int32_t count, void** flags_out) {
    MB_CTX(ctx);
    if (count <= 0 || !flags_out) return fail(MB_ERR_INVALID_ARG, "mb_flags_alloc: bad argument");
    // a private cudaMalloc (not a sub-allocation of somebody's pool), so the exported handle maps exactly this array
    MB_CUDA(cudaMalloc(flags_out, sizeof(unsigned long long) * (size_t)count));
    MB_CUDA(cudaMemset(*flags_out, 0, sizeof(unsigned long long) * (size_t)count));
    MB_CUDA(cudaDeviceSynchronize());
    return MB_OK;
}
int32_t mb_flags_free(mb_ctx* ctx, void* flags) {
    MB_CTX(ctx);
    if (flags) cudaFree(flags);
    return MB_OK;
}
int32_t mb_flag_signal(mb_ctx* ctx, void* flag, int64_t value) {
    MB_CTX(ctx);
    if (!flag) return fail(MB_ERR_INVALID_ARG, "mb_flag_signal: null flag");
    MB_CUDA(mb::flag_signal(flag, (unsigned long long)value, ctx->stream));
    ctx->launches++;
    return MB_OK;
}
int32_t mb_flag_wait(mb_ctx* ctx, const void* flag, int64_t value) {
    MB_CTX(ctx);
    if (!flag) return fail(MB_ERR_INVALID_ARG, "mb_flag_wait: null flag");
    MB_CUDA(mb::flag_wait(flag, (unsigned long long)value, ctx->stream));
    ctx->launches++;
    return MB_OK;
}
int32_t mb_memcpy_async(mb_ctx* ctx, void* dst, const void* src, int64_t bytes) {
    MB_CTX(ctx);
    if (bytes < 0 || (bytes > 0 && (!dst || !src))) return fail(MB_ERR_INVALID_ARG, "mb_memcpy_async: bad argument");
    if (bytes == 0) return MB_OK;
    MB_CUDA(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return MB_OK;
}

// ----------------------------------------------------------------------------- elementwise
int32_t mb_block_add(mb_ctx* ctx, const mb_block* A, const mb_block* B, mb_block* out) { return binary_op(ctx, mb::EW_ADD, A, B, out, "add"); }
int32_t mb_block_sub(mb_ctx* ctx, const mb_block* A, const mb_block* B, mb_block* out) { return binary_op(ctx, mb::EW_SUB, A, B, out, "subtract"); }
int32_t mb_block_hadamard(mb_ctx* ctx, const mb_block* A, const mb_block* B, mb_block* out) { return binary_op(ctx, mb::EW_MUL, A, B, out, "dotProduct"); }
int32_t mb_block_axpb(mb_ctx* ctx, const mb_block* A, double alpha, double beta, mb_block* out) {
    return unary_op(ctx, mb::EW_AXPB, A, out, alpha, beta, "axpb");
}
int32_t mb_block_fill(mb_ctx* ctx, mb_block* blk, double value) {
    return unary_op(ctx, mb::EW_FILL, blk, blk, 0.0, value, "fill");
}
int32_t mb_block_div(mb_ctx* ctx, const mb_block* A, double b, int32_t b_over_a, mb_block* out) {
    return unary_op(ctx, b_over_a ? mb::EW_RDIV : mb::EW_DIV, A, out, b, 0.0, "divide");
}

int32_t mb_block_copy(mb_ctx* ctx, const mb_block* A, mb_block* out) {
    MB_CTX(ctx);
    if (!A || !out) return fail(MB_ERR_INVALID_ARG, "mb_block_copy: null block");
    int32_t r = same_shape(A, out, "copy");
    if (r) return r;
    return copy_convert(ctx, A, out);
}

int32_t mb_block_transpose(mb_ctx* ctx, const mb_block* A, mb_block* out) {
    MB_CTX(ctx);
    if (!A || !out) return fail(MB_ERR_INVALID_ARG, "mb_block_transpose: null block");
    if (out->rows != A->cols || out->cols != A->rows)
        return fail(MB_ERR_DIM_MISMATCH, "transpose: result block is %dx%d, expected %dx%d", out->rows, out->cols, A->cols, A->rows);
    mb_block view = *A;     // A^T as a view, then materialise it (denseBlock.t.copy)
    view.owns = 0;
    std::swap(view.rows, view.cols);
    view.is_transpose = !A->is_transpose;
    return copy_convert(ctx, &view, out);
}

int32_t mb_block_sum(mb_ctx* ctx, const mb_block* A, double* sum_out) {
    MB_CTX(ctx);
    MB_LOCK(ctx);
    if (!A || !sum_out) return fail(MB_ERR_INVALID_ARG, "mb_block_sum: null argument");
    if (A->dtype != MB_F64) return fail(MB_ERR_UNSUPPORTED, "mb_block_sum: fp64 blocks only");
    if (A->rows == 0 || A->cols == 0) { *sum_out = 0.0; return MB_OK; }
    const int minor = A->is_transpose ? A->cols : A->rows, major = A->is_transpose ? A->rows : A->cols;
    MB_CUDA(mb::sum_f64(f64_ptr(A), minor, major, A->ld, ctx->scratch, ctx->stream));
    ctx->launches += 2;
    MB_CUDA(cudaMemcpyAsync(ctx->host_scalar, ctx->scratch, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(cudaStreamSynchronize(ctx->stream));
    *sum_out = *ctx->host_scalar;
    return MB_OK;
}

int32_t mb_block_gemv(mb_ctx* ctx, const mb_block* A, const mb_block* x, mb_block* y, int32_t accumulate) {
    MB_CTX(ctx);
    MB_LOCK(ctx);
    if (!A || !x || !y) return fail(MB_ERR_INVALID_ARG, "mb_block_gemv: null block");
    vec_view xv, yv;
    if (A->dtype != MB_F64 || !as_vector(x, &xv) || !as_vector(y, &yv))
        return fail(MB_ERR_UNSUPPORTED, "mb_block_gemv: fp64 matrix and fp64 single-column (or single-row) vectors only");
    if (A->cols != xv.len)
        return fail(MB_ERR_DIM_MISMATCH, "Dimension mismatch during matrix-vector multiplication: %d vs %d", A->cols, xv.len);
    if (A->rows != yv.len)
        return fail(MB_ERR_DIM_MISMATCH, "mb_block_gemv: result vector has %d elements, expected %d", yv.len, A->rows);
    // a transposed view is the column-major (cols x rows) array underneath: y = S^T x
    const bool trans = A->is_transpose != 0;
    const int m = trans ? A->cols : A->rows, n = trans ? A->rows : A->cols;
    const size_t need = mb::gemv_workspace_doubles(trans, m, n);
    if (need > ctx->vec_ws_doubles) {
        if (ctx->vec_ws) { MB_CUDA(cudaStreamSynchronize(ctx->stream)); MB_CUDA(cudaFree(ctx->vec_ws)); ctx->vec_ws = nullptr; ctx->vec_ws_doubles = 0; }
        MB_CUDA(cudaMalloc(&ctx->vec_ws, need * sizeof(double)));
        ctx->vec_ws_doubles = need;
    }
    int launches = 0;
    MB_CUDA(mb::gemv_f64(trans, m, n, f64_ptr(A), A->ld, xv.p, xv.inc, yv.p, yv.inc, accumulate != 0, ctx->vec_ws, ctx->stream,
                         &launches));
    ctx->launches += launches;
    return MB_OK;
}

int32_t mb_block_dot(mb_ctx* ctx, const mb_block* x, const mb_block* y, double* dot_out) {
    MB_CTX(ctx);
    MB_LOCK(ctx);
    if (!x || !y || !dot_out) return fail(MB_ERR_INVALID_ARG, "mb_block_dot: null argument");
    vec_view xv, yv;
    if (!as_vector(x, &xv) || !as_vector(y, &yv))
        return fail(MB_ERR_UNSUPPORTED, "mb_block_dot: fp64 single-column (or single-row) vectors only");
    if (xv.len != yv.len)
        return fail(MB_ERR_DIM_MISMATCH, "the length of these two vectors are not the same: %d vs %d", xv.len, yv.len);
    if (xv.len == 0) { *dot_out = 0.0; return MB_OK; }
    MB_CUDA(mb::dot_f64(xv.len, xv.p, xv.inc, yv.p, yv.inc, ctx->scratch, ctx->stream));
    ctx->launches += 2;
    MB_CUDA(cudaMemcpyAsync(ctx->host_scalar, ctx->scratch, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(cudaStreamSynchronize(ctx->stream));
    *dot_out = *ctx->host_scalar;
    return MB_OK;
}

int32_t mb_block_ger(mb_ctx* ctx, const mb_block* x, const mb_block* y, mb_block* out) {
    MB_CTX(ctx);
    if (!x || !y || !out) return fail(MB_ERR_INVALID_ARG, "mb_block_ger: null block");
    vec_view xv, yv;
    if (out->dtype != MB_F64 || !as_vector(x, &xv) || !as_vector(y, &yv))
        return fail(MB_ERR_UNSUPPORTED, "mb_block_ger: fp64 vectors and an fp64 result block only");
    if (out->rows != xv.len || out->cols != yv.len)
        return fail(MB_ERR_DIM_MISMATCH, "mb_block_ger: result block is %dx%d, expected %dx%d", out->rows, out->cols, xv.len, yv.len);
    if (out->is_transpose) std::swap(xv, yv);       // (x y^T)^T = y x^T in the array underneath
    MB_CUDA(mb::ger_f64(xv.len, yv.len, xv.p, xv.inc, yv.p, yv.inc, f64_ptr(out), out->ld, ctx->stream));
    ctx->launches++;
    return MB_OK;
}

// ---------------------------------------------------------------------- factorizations (SURVEY 8 f4)
static int32_t int_scratch(mb_ctx* ctx, size_t count) {
    if (count > ctx->int_ws_count) {
        if (ctx->int_ws) { MB_CUDA(cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->int_ws); ctx->int_ws = nullptr; ctx->int_ws_count = 0; }
        MB_CUDA(cudaMalloc(&ctx->int_ws, count * sizeof(int)));
        ctx->int_ws_count = count;
    }
    if (count > ctx->int_host_count) {
        if (ctx->int_host) { cudaFreeHost(ctx->int_host); ctx->int_host = nullptr; ctx->int_host_count = 0; }
        MB_CUDA(cudaMallocHost(&ctx->int_host, count * sizeof(int)));
        ctx->int_host_count = count;
    }
    return MB_OK;
}
static mb::FView fview(const mb_block* b) { return mb::FView{f64_ptr(b), rs(b), cs(b), b->rows, b->cols}; }

int32_t mb_block_lu(mb_ctx* ctx, mb_block* A, int32_t* perm_out) {
    MB_CTX(ctx);
    MB_LOCK(ctx);
    if (!A) return fail(MB_ERR_INVALID_ARG, "mb_block_lu: null block");
    if (A->dtype != MB_F64) return fail(MB_ERR_UNSUPPORTED, "mb_block_lu: fp64 blocks only");
    const int m = A->rows, n = A->cols;
    if (m == 0 || n == 0) return MB_OK;
    int32_t r = int_scratch(ctx, (size_t)2 * m + 8);
    if (r) return r;
    int *piv = ctx->int_ws, *perm = ctx->int_ws + m, *info = ctx->int_ws + 2 * m;
    int launches = 0;
    // rows that are never a pivot position keep themselves: start from the identity interchange
    std::vector<int> ident(m);
    for (int i = 0; i < m; ++i) ident[i] = i;
    std::memcpy(ctx->int_host, ident.data(), sizeof(int) * m);
    MB_CUDA(cudaMemcpyAsync(piv, ctx->int_host, sizeof(int) * m, cudaMemcpyHostToDevice, ctx->stream));
    MB_CUDA(cudaStreamSynchronize(ctx->stream));
    MB_CUDA(mb::getrf(fview(A), piv, nullptr, info, ctx->num_sms, ctx->stream, &launches));
    ctx->launches += launches;
    MB_CUDA(cudaMemcpyAsync(ctx->int_host, piv, sizeof(int) * (2 * (size_t)m + 1), cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (perm_out) {
        // the reference's pArray (matrix/DenseVecMatrix.scala:303-308): apply the interchanges to 0..m-1
        for (int i = 0; i < m; ++i) perm_out[i] = i;
        for (int i = 0; i < std::min(m, n); ++i) std::swap(perm_out[i], perm_out[ctx->int_host[i]]);
    }
    (void)perm;
    // like Breeze's LU (dgetrf), an exactly singular pivot is not an error here: U carries the zero
    return MB_OK;
}

int32_t mb_block_cholesky(mb_ctx* ctx, mb_block* A) {
    MB_CTX(ctx);
    MB_LOCK(ctx);
    if (!A) return fail(MB_ERR_INVALID_ARG, "mb_block_cholesky: null block");
    if (A->dtype != MB_F64) return fail(MB_ERR_UNSUPPORTED, "mb_block_cholesky: fp64 blocks only");
    if (A->rows != A->cols) return fail(MB_ERR_DIM_MISMATCH, "Cholesky needs a square matrix: %d x %d", A->rows, A->cols);
    if (A->rows == 0) return MB_OK;
    int32_t r = int_scratch(ctx, 8);
    if (r) return r;
    int launches = 0;
    MB_CUDA(mb::potrf_lower(fview(A), ctx->int_ws, ctx->num_sms, ctx->stream, &launches));
    ctx->launches += launches;
    MB_CUDA(cudaMemcpyAsync(ctx->int_host, ctx->int_ws, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ctx->int_host[0] != 0)      // Breeze: NotConvergedException / MatrixNotSymmetricException family -> RuntimeException
        return fail(MB_ERR_CUDA, "Cholesky: the matrix is not positive definite (leading minor %d)", ctx->int_host[0]);
    return MB_OK;
}

int32_t mb_block_inverse(mb_ctx* ctx, const mb_block* A, mb_block* out) {
    MB_CTX(ctx);
    MB_LOCK(ctx);
    if (!A || !out) return fail(MB_ERR_INVALID_ARG, "mb_block_inverse: null block");
    if (A->dtype != MB_F64 || out->dtype != MB_F64) return fail(MB_ERR_UNSUPPORTED, "mb_block_inverse: fp64 blocks only");
    if (A->rows != A->cols) return fail(MB_ERR_DIM_MISMATCH, "Inversion only support square matrix: %d v.s %d", A->rows, A->cols);
    if (out->rows != A->rows || out->cols != A->cols) return fail(MB_ERR_DIM_MISMATCH, "mb_block_inverse: result block is %dx%d", out->rows, out->cols);
    const int n = A->rows;
    if (n == 0) return MB_OK;
    int32_t r = int_scratch(ctx, (size_t)2 * n + 8);
    if (r) return r;
    // working copy of A for the factors (packed, even leading dimension)
    const int ld = (n + 1) & ~1;
    double* lu = nullptr;
    MB_CUDA(cudaMalloc(&lu, (size_t)ld * n * sizeof(double)));
    mb_block tmp;
    tmp.data = lu; tmp.rows = n; tmp.cols = n; tmp.ld = ld; tmp.dtype = MB_F64; tmp.device = ctx->device;
    r = copy_convert(ctx, A, &tmp);
    if (r) { cudaFree(lu); return r; }
    int *piv = ctx->int_ws, *info = ctx->int_ws + 2 * n;
    int launches = 0;
    cudaError_t e = mb::getrf(fview(&tmp), piv, nullptr, info, ctx->num_sms, ctx->stream, &launches);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->int_host, info, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess && ctx->int_host[0] != 0) {
        cudaFree(lu);
        return fail(MB_ERR_CUDA, "matrix is singular (zero pivot in column %d)", ctx->int_host[0] - 1);   // Breeze: MatrixSingularException
    }
    if (e == cudaSuccess) e = mb::inverse_from_lu(fview(&tmp), piv, fview(out), ctx->num_sms, ctx->stream, &launches);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(lu);
    ctx->launches += launches;
    if (e != cudaSuccess) return cuda_fail(e, "mb_block_inverse");
    return MB_OK;
}

int32_t mb_block_trsm(mb_ctx* ctx, const mb_block* T, int32_t lower, int32_t unit_diagonal, mb_block* B) {
    MB_CTX(ctx);
    if (!T || !B) return fail(MB_ERR_INVALID_ARG, "mb_block_trsm: null block");
    if (T->dtype != MB_F64 || B->dtype != MB_F64) return fail(MB_ERR_UNSUPPORTED, "mb_block_trsm: fp64 blocks only");
    if (T->rows != T->cols || T->rows != B->rows)
        return fail(MB_ERR_DIM_MISMATCH, "mb_block_trsm: triangle is %dx%d, right-hand side has %d rows", T->rows, T->cols, B->rows);
    int launches = 0;
    MB_CUDA(mb::trsm_left(fview(T), lower != 0, unit_diagonal != 0, fview(B), ctx->num_sms, ctx->stream, &launches));
    ctx->launches += launches;
    return MB_OK;
}

int32_t mb_fill_uniform(mb_ctx* ctx, mb_block* blk, int64_t partition_seed, int64_t first, double lo, double hi,
                        int32_t row_major) {
    MB_CTX(ctx);
    if (!blk || first < 0) return fail(MB_ERR_INVALID_ARG, "mb_fill_uniform: bad argument");
    if (blk->dtype != MB_F64) return fail(MB_ERR_UNSUPPORTED, "mb_fill_uniform: fp64 blocks only (convert afterwards)");
    // generator.setSeed(partition.seed) -> XORShiftRandom.setSeed -> seed = hashSeed(s)
    const unsigned long long state0 = (unsigned long long)mb_hash_seed(partition_seed);
    int launches = 0;
    MB_CUDA(mb::fill_uniform_f64(f64_ptr(blk), rs(blk), cs(blk), blk->rows, blk->cols, row_major ? 1 : 0, state0, first, lo,
                                 hi, ctx->stream, &launches));
    ctx->launches += launches;
    return MB_OK;
}

// ---------------------------------------------------------------------------------- sparse blocks
// `new SubMatrix(spMatrix = ...)` (matrix/SubMatrix.scala:22-25): CSC device arrays; see include/marlin_b200.h.
static int32_t spblock_alloc(mb_ctx* ctx, int32_t rows, int32_t cols, long long nnz, mb_spblock** out) {
    mb_spblock* sp = new (std::nothrow) mb_spblock();
    if (!sp) return fail(MB_ERR_OOM, "host allocation failed");
    sp->rows = rows; sp->cols = cols; sp->nnz = nnz; sp->device = ctx->device;
    cudaError_t e = cudaMalloc(&sp->col_ptr, sizeof(int) * ((size_t)cols + 1));
    if (e == cudaSuccess && nnz > 0) e = cudaMalloc(&sp->row_idx, sizeof(int) * (size_t)nnz);
    if (e == cudaSuccess && nnz > 0) e = cudaMalloc(&sp->val, sizeof(double) * (size_t)nnz);
    if (e != cudaSuccess) { mb_spblock_free(ctx, sp); *out = nullptr; return cuda_fail(e, "cudaMalloc(sparse block)"); }
    *out = sp;
    return MB_OK;
}

static int32_t dense_f64(const mb_block* b, const char* what) {
    if (b->dtype != MB_F64) return fail(MB_ERR_UNSUPPORTED, "%s: fp64 dense blocks only", what);
    return MB_OK;
}

static int32_t check_out(const mb_block* C, int rows, int cols, const char* what) {
    if (!C) return fail(MB_ERR_INVALID_ARG, "%s: null result block", what);
    if (C->dtype != MB_F64) return fail(MB_ERR_UNSUPPORTED, "%s: the result block must be fp64", what);
    if (C->rows != rows || C->cols != cols)
        return fail(MB_ERR_DIM_MISMATCH, "%s: result block is %dx%d, expected %dx%d", what, C->rows, C->cols, rows, cols);
    return MB_OK;
}

// per-call workspace of the tile pointers of the scatter products: stream-ordered, released on the same stream
struct tile_ws {
    int* p = nullptr;
    cudaStream_t st;
    ~tile_ws() { if (p) cudaFreeAsync(p, st); }
};

int32_t mb_spblock_upload(mb_ctx* ctx, int32_t rows, int32_t cols, const int32_t* col_ptr, const int32_t* row_idx,
                          const double* val, mb_spblock** out) {
    MB_CTX(ctx);
    if (!out) return fail(MB_ERR_INVALID_ARG, "mb_spblock_upload: null output");
    int32_t r = mb_csc_check(rows, cols, col_ptr, row_idx);
    if (r) return r;
    const long long nnz = col_ptr[cols];
    if (nnz > 0 && !val) return fail(MB_ERR_INVALID_ARG, "mb_spblock_upload: null values");
    r = spblock_alloc(ctx, rows, cols, nnz, out);
    if (r) return r;
    mb_spblock* sp = *out;
    cudaError_t e = cudaMemcpyAsync(sp->col_ptr, col_ptr, sizeof(int) * ((size_t)cols + 1), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && nnz > 0)
        e = cudaMemcpyAsync(sp->row_idx, row_idx, sizeof(int) * (size_t)nnz, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && nnz > 0)
        e = cudaMemcpyAsync(sp->val, val, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { mb_spblock_free(ctx, sp); *out = nullptr; return cuda_fail(e, "mb_spblock_upload"); }
    return MB_OK;
}

int32_t mb_spblock_download(mb_ctx* ctx, const mb_spblock* sp, int32_t* col_ptr, int32_t* row_idx, double* val) {
    MB_CTX(ctx);
    if (!sp || !col_ptr || (sp->nnz > 0 && (!row_idx || !val))) return fail(MB_ERR_INVALID_ARG, "mb_spblock_download: null argument");
    MB_CUDA(cudaMemcpyAsync(col_ptr, sp->col_ptr, sizeof(int) * ((size_t)sp->cols + 1), cudaMemcpyDeviceToHost, ctx->stream));
    if (sp->nnz > 0) {
        MB_CUDA(cudaMemcpyAsync(row_idx, sp->row_idx, sizeof(int) * (size_t)sp->nnz, cudaMemcpyDeviceToHost, ctx->stream));
        MB_CUDA(cudaMemcpyAsync(val, sp->val, sizeof(double) * (size_t)sp->nnz, cudaMemcpyDeviceToHost, ctx->stream));
    }
    MB_CUDA(cudaStreamSynchronize(ctx->stream));
    return MB_OK;
}

int32_t mb_spblock_info(const mb_spblock* sp, int32_t* rows, int32_t* cols, int64_t* nnz) {
    if (!sp) return fail(MB_ERR_INVALID_ARG, "null sparse block");
    if (rows) *rows = sp->rows;
    if (cols) *cols = sp->cols;
    if (nnz) *nnz = sp->nnz;
    return MB_OK;
}

int32_t mb_spblock_free(mb_ctx* ctx, mb_spblock* sp) {
    if (!sp) return MB_OK;
    if (ctx) cudaSetDevice(ctx->device);
    cudaFree(sp->col_ptr);
    cudaFree(sp->row_idx);
    cudaFree(sp->val);
    delete sp;
    return MB_OK;
}

int32_t mb_spblock_copy(mb_ctx* ctx, const mb_spblock* sp, mb_spblock** out) {
    MB_CTX(ctx);
    if (!sp || !out) return fail(MB_ERR_INVALID_ARG, "mb_spblock_copy: null argument");
    int32_t r = spblock_alloc(ctx, sp->rows, sp->cols, sp->nnz, out);
    if (r) return r;
    mb_spblock* d = *out;
    cudaError_t e = cudaMemcpyAsync(d->col_ptr, sp->col_ptr, sizeof(int) * ((size_t)sp->cols + 1), cudaMemcpyDeviceToDevice,
                                    ctx->stream);
    if (e == cudaSuccess && sp->nnz > 0)
        e = cudaMemcpyAsync(d->row_idx, sp->row_idx, sizeof(int) * (size_t)sp->nnz, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess && sp->nnz > 0)
        e = cudaMemcpyAsync(d->val, sp->val, sizeof(double) * (size_t)sp->nnz, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e != cudaSuccess) { mb_spblock_free(ctx, d); *out = nullptr; return cuda_fail(e, "mb_spblock_copy"); }
    return MB_OK;
}

int32_t mb_spblock_values(mb_ctx* ctx, mb_spblock* sp, mb_block** out) {
    if (!sp) return fail(MB_ERR_INVALID_ARG, "null sparse block");
    return mb_block_wrap(ctx, sp->val, 0, int32_t(sp->nnz), 1, int32_t(sp->nnz > 0 ? sp->nnz : 1), 0, MB_F64, out);
}

int32_t mb_spblock_to_dense(mb_ctx* ctx, const mb_spblock* sp, mb_block* out) {
    MB_CTX(ctx);
    if (!sp) return fail(MB_ERR_INVALID_ARG, "mb_spblock_to_dense: null sparse block");
    int32_t r = check_out(out, sp->rows, sp->cols, "toDense");
    if (r) return r;
    int launches = 0;
    MB_CUDA(mb::sparse_to_dense(sp->col_ptr, sp->row_idx, sp->val, sp->rows, sp->cols, f64_ptr(out), rs(out), cs(out),
                                ctx->stream, &launches));
    ctx->launches += launches;
    return MB_OK;
}

int32_t mb_spblock_rand(mb_ctx* ctx, int32_t rows, int32_t cols, double sparsity, int64_t partition_seed, mb_spblock** out) {
    MB_CTX(ctx);
    if (!out) return fail(MB_ERR_INVALID_ARG, "mb_spblock_rand: null output");
    int32_t count = 0;
    int32_t r = mb_sparse_rand_count(rows, cols, sparsity, &count);
    if (r) return r;
    r = spblock_alloc(ctx, rows, cols, (long long)count * cols, out);
    if (r) return r;
    int launches = 0;
    cudaError_t e = mb::sparse_rand(rows, cols, count, (unsigned long long)partition_seed, (*out)->col_ptr, (*out)->row_idx,
                                    (*out)->val, ctx->stream, &launches);
    ctx->launches += launches;
    if (e != cudaSuccess) { mb_spblock_free(ctx, *out); *out = nullptr; return cuda_fail(e, "mb_spblock_rand"); }
    return MB_OK;
}

int32_t mb_spmm_dense_sparse(mb_ctx* ctx, const mb_block* A, const mb_spblock* B, mb_block* C, int32_t accumulate) {
    MB_CTX(ctx);
    if (!A || !B) return fail(MB_ERR_INVALID_ARG, "multDenseSparse: null operand");
    if (A->cols != B->rows) return fail(MB_ERR_DIM_MISMATCH, "matrix dimension mismatch: %d v.s %d", A->cols, B->rows);
    int32_t r = dense_f64(A, "multDenseSparse");
    if (r) return r;
    if ((r = check_out(C, A->rows, B->cols, "multDenseSparse"))) return r;
    int launches = 0;
    MB_CUDA(mb::spmm_dense_sparse(f64_ptr(A), rs(A), cs(A), A->rows, B->col_ptr, B->row_idx, B->val, B->cols, f64_ptr(C), rs(C),
                                  cs(C), accumulate ? 1 : 0, ctx->stream, &launches));
    ctx->launches += launches;
    return MB_OK;
}

int32_t mb_spmm_sparse_dense(mb_ctx* ctx, const mb_spblock* A, const mb_block* B, mb_block* C, int32_t accumulate) {
    MB_CTX(ctx);
    if (!A || !B) return fail(MB_ERR_INVALID_ARG, "multSparseDense: null operand");
    if (A->cols != B->rows) return fail(MB_ERR_DIM_MISMATCH, "matrix dimension mismatch: %d v.s %d", A->cols, B->rows);
    int32_t r = dense_f64(B, "multSparseDense");
    if (r) return r;
    if ((r = check_out(C, A->rows, B->cols, "multSparseDense"))) return r;
    tile_ws ws;
    ws.st = ctx->stream;
    const long long need = mb::sparse_tile_ptr_ints(A->rows, A->cols);
    if (need > 0 && B->cols > 0) MB_CUDA(cudaMallocAsync(&ws.p, sizeof(int) * (size_t)need, ctx->stream));
    int launches = 0;
    MB_CUDA(mb::spmm_sparse_dense(A->col_ptr, A->row_idx, A->val, A->rows, A->cols, f64_ptr(B), rs(B), cs(B), B->cols, f64_ptr(C),
                                  rs(C), cs(C), accumulate ? 1 : 0, ws.p, ctx->stream, &launches));
    ctx->launches += launches;
    return MB_OK;
}

int32_t mb_spgemm_to_dense(mb_ctx* ctx, const mb_spblock* A, const mb_spblock* B, mb_block* C, int32_t accumulate) {
    MB_CTX(ctx);
    if (!A || !B) return fail(MB_ERR_INVALID_ARG, "SparseMatrix.multiply: null operand");
    if (A->cols != B->rows) return fail(MB_ERR_DIM_MISMATCH, "matrix dimension mismatch: %d v.s %d", A->cols, B->rows);
    int32_t r = check_out(C, A->rows, B->cols, "SparseMatrix.multiply");
    if (r) return r;
    tile_ws ws;
    ws.st = ctx->stream;
    const long long need = mb::sparse_tile_ptr_ints(A->rows, A->cols);
    if (need > 0 && B->cols > 0) MB_CUDA(cudaMallocAsync(&ws.p, sizeof(int) * (size_t)need, ctx->stream));
    int launches = 0;
    MB_CUDA(mb::spgemm_to_dense(A->col_ptr, A->row_idx, A->val, A->rows, A->cols, B->col_ptr, B->row_idx, B->val, B->cols,
                                f64_ptr(C), rs(C), cs(C), accumulate ? 1 : 0, ws.p, ctx->stream, &launches));
    ctx->launches += launches;
    return MB_OK;
}

}  // extern "C"

