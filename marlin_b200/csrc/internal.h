// Internal definitions shared by the translation units behind the C ABI (capi.cu, dist.cu): the context and block
// records, error plumbing and small helpers.  Not installed; include/marlin_b200.h is the public surface.
#pragma once
#include "../../include/marlin_b200.h"

#include <cuda_runtime.h>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <mutex>

struct mb_ctx {
    int device = 0;
    int num_sms = 148;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    std::atomic<long long> launches{0};
    double* scratch = nullptr;          // sum partials + result
    double* host_scalar = nullptr;      // pinned
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // pipelined host<->device path (mb_matmul_blocked_host): copy streams + a grow-only device workspace
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    void* workspace = nullptr;
    size_t workspace_bytes = 0;
    // fp64 mode (mb_set_fp64_mode) and the digit-plane workspace of the int8-split path
    int fp64_mode = MB_FP64_NATIVE;
    int fp64_slices = 7;
    int fp64_bits = 7;
    void* ozaki_ws = nullptr;
    size_t ozaki_ws_bytes = 0;
    // partial vectors of the matrix x vector kernels (grow-only)
    double* vec_ws = nullptr;
    size_t vec_ws_doubles = 0;
    // pivots / permutation / info of the factorization entries (grow-only) + a pinned mirror for the results
    int* int_ws = nullptr;
    size_t int_ws_count = 0;
    int* int_host = nullptr;
    size_t int_host_count = 0;
    // Entry points that use the context's own scratch buffers, workspaces, events or copy streams take this lock, so
    // threads sharing one context (Spark local[N] task threads) serialise there; kernel-only entries (gemm, element-wise,
    // transpose, fill) touch no shared host state and need none.  Threads that want concurrency use one context each.
    std::recursive_mutex mu;
};

struct mb_block {
    void* data = nullptr;      // device base pointer (element 0 of the underlying array)
    long long offset = 0;      // in elements
    int rows = 0, cols = 0;    // logical dims
    int ld = 0;                // majorStride
    int is_transpose = 0;
    int dtype = MB_F64;
    int owns = 0;
    int device = 0;
    void* ready_event = nullptr;   // optional cudaEvent_t: the block's contents are final once it has completed
};

// CSC sparse block (include/marlin_b200.h): device arrays owned by the record; row_idx / val are null when nnz == 0
struct mb_spblock {
    int rows = 0, cols = 0;
    long long nnz = 0;
    int* col_ptr = nullptr;
    int* row_idx = nullptr;
    double* val = nullptr;
    int device = 0;
};

namespace mb {
cudaError_t ipc_export(const void* dptr, unsigned char handle[64], long long* offset, long long* alloc_bytes);
cudaError_t ipc_open(const unsigned char handle[64], void** base_out);
cudaError_t ipc_open_ex(const unsigned char handle[64], void** base_out, bool pinned);
unsigned long long ipc_evictions();
cudaError_t ipc_close(const unsigned char handle[64]);
cudaError_t ipc_close_all();
cudaError_t flag_signal(void* flag, unsigned long long v, cudaStream_t st);
bool stream_memops_available();
cudaError_t stream_write64(void* flag, unsigned long long v, cudaStream_t st);
cudaError_t stream_wait64_geq(const void* flag, unsigned long long v, cudaStream_t st);
cudaError_t flag_wait(const void* flag, unsigned long long v, cudaStream_t st);
cudaError_t flag_wait_bounded(const void* flag, unsigned long long v, long long timeout_ns, unsigned long long* status,
                              cudaStream_t st, unsigned long long tag = 0);
}  // namespace mb

// thread-local message of the last failing call (defined in capi.cu)
int32_t mb_fail(int32_t code, const char* fmt, ...);
#define fail mb_fail
inline int32_t cuda_fail(cudaError_t e, const char* what) {
    return fail(e == cudaErrorMemoryAllocation ? MB_ERR_OOM : MB_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}
#define MB_CUDA(call)                                       \
    do {                                                    \
        cudaError_t _e = (call);                            \
        if (_e != cudaSuccess) return cuda_fail(_e, #call); \
    } while (0)

inline size_t elem_size(int dtype) { return dtype == MB_F64 ? 8 : (dtype == MB_F32 ? 4 : 2); }
inline char* elem_ptr(const mb_block* b) { return static_cast<char*>(b->data) + b->offset * (long long)elem_size(b->dtype); }
inline double* f64_ptr(const mb_block* b) { return reinterpret_cast<double*>(elem_ptr(b)); }
// strides of the logical (rows x cols) view
inline long long rs(const mb_block* b) { return b->is_transpose ? b->ld : 1; }
inline long long cs(const mb_block* b) { return b->is_transpose ? 1 : b->ld; }

inline int32_t check_ctx(mb_ctx* ctx) {
    if (!ctx) return fail(MB_ERR_INVALID_ARG, "null context");
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    return MB_OK;
}
#define MB_CTX(ctx)                        \
    do {                                   \
        int32_t _r = check_ctx(ctx);       \
        if (_r != MB_OK) return _r;        \
    } while (0)
#define MB_LOCK(ctx) std::lock_guard<std::recursive_mutex> _mb_lock((ctx)->mu)

