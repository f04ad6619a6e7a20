/*
 * marlin_b200.h — C ABI of libmarlin_b200.so, the B200 (sm_100a) drop-in for the dense
 * block-matrix hot path of PasaLab/marlin (edu.nju.pasalab.marlin.matrix).
 *
 * The reference has no FFI of its own; its only native seam is Breeze -> netlib-java
 * BLAS.dgemm (third-party, not in the tree).  The entry points below are what a JNI veneer
 * for edu.nju.pasalab.marlin.matrix.{SubMatrix,BlockMatrix,DenseVecMatrix} and
 * edu.nju.pasalab.marlin.utils.MTUtils would bind (see INTEGRATION.md for the Scala/JNI side).
 * Every entry cites the reference code it replaces (paths relative to the reference's
 * src/main/scala/edu/nju/pasalab/marlin/).
 *
 * Conventions
 *   - plain C, no torch / C++ types; all functions return int32 status (0 = MB_OK, <0 = error);
 *     mb_last_error() returns a thread-local message for the last failing call.
 *   - one mb_ctx per process and GPU (one process per GPU, like one Spark executor per device).
 *   - a block (mb_block) is the device-resident analogue of SubMatrix.denseBlock: Breeze
 *     DenseMatrix semantics (data, offset, rows, cols, majorStride, isTranspose), column-major:
 *        element(r,c) = data[offset + r + c*ld]            if !is_transpose
 *                     = data[offset + c + r*ld]            if  is_transpose
 *   - there is NO CPU fallback: without a CUDA device every compute entry returns MB_ERR_CUDA.
 */
#ifndef MARLIN_B200_H
#define MARLIN_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

#define MB_OK                 0
#define MB_ERR_INVALID_ARG   -1   /* -> IllegalArgumentException on the JVM side            */
#define MB_ERR_DIM_MISMATCH  -2   /* -> IllegalArgumentException ("Dimension mismatch ...")  */
#define MB_ERR_UNSUPPORTED   -3   /* -> IllegalArgumentException ("currently not supported") */
#define MB_ERR_CUDA          -4   /* -> RuntimeException                                     */
#define MB_ERR_OOM           -5
#define MB_ERR_EMPTY         -6   /* -> RuntimeException (empty RDD: DistributedMatrixSuite "empty rows") */

typedef enum { MB_F64 = 0, MB_BF16 = 1, MB_F32 = 2 } mb_dtype;

typedef struct mb_ctx   mb_ctx;
typedef struct mb_block mb_block;

/* ---- lifetime (SparkContext lifetime in the reference) --------------------------------- */
int32_t     mb_init(int32_t device, mb_ctx** out);
int32_t     mb_shutdown(mb_ctx* ctx);
const char* mb_last_error(void);
const char* mb_version(void);
/* Use an externally owned stream (e.g. torch's current stream) for every later call.  The handle is
 * used as CUDA would: NULL is the legacy default stream.  mb_reset_stream returns to the ctx's own
 * (non-blocking) stream, which is what a fresh ctx uses. */
int32_t     mb_set_stream(mb_ctx* ctx, void* cuda_stream);
int32_t     mb_reset_stream(mb_ctx* ctx);
int32_t     mb_synchronize(mb_ctx* ctx);
/* Number of kernels this library has launched on ctx since init (bench.py's gpu_launches). */
int64_t     mb_launch_count(mb_ctx* ctx);
/* CUDA-event timing on the ctx stream, so callers can time kernels on the launching stream. */
int32_t     mb_timer_start(mb_ctx* ctx);
int32_t     mb_timer_stop(mb_ctx* ctx, float* ms_out);

/* ---- blocks: `new SubMatrix(denseMatrix = ...)` (matrix/SubMatrix.scala:16-20) ---------- */
int32_t mb_block_alloc(mb_ctx* ctx, int32_t rows, int32_t cols, mb_dtype dtype, mb_block** out);
/* Non-owning view over device memory someone else allocated (torch tensor, NCCL buffer). */
int32_t mb_block_wrap(mb_ctx* ctx, void* device_ptr, int64_t offset, int32_t rows, int32_t cols,
                      int32_t ld, int32_t is_transpose, mb_dtype dtype, mb_block** out);
/* Host fp64 (Breeze data/offset/majorStride/isTranspose) -> packed device block (ld = rows),
 * optionally rounded to bf16 (round-to-nearest-even) for the bf16 path. */
int32_t mb_block_upload(mb_ctx* ctx, const double* host, int64_t offset, int32_t rows, int32_t cols,
                        int32_t ld, int32_t is_transpose, mb_dtype store_as, mb_block** out);
/* toBreeze()/collect (matrix/BlockMatrix.scala:70-85): packed column-major fp64, leading dim ld. */
int32_t mb_block_download(mb_ctx* ctx, const mb_block* blk, double* host, int32_t ld);
int32_t mb_block_free(mb_ctx* ctx, mb_block* blk);
int32_t mb_block_info(const mb_block* blk, int32_t* rows, int32_t* cols, int32_t* ld,
                      int32_t* is_transpose, int32_t* dtype, void** device_ptr);
/* Optional: a cudaEvent_t that completes when the block's contents are final (blocks are immutable values, like the
 * blocks of a cached RDD).  mb_matmul_blocked_dist then offers such tiles to the other ranks as soon as that event has
 * completed instead of after everything queued on the ctx stream — the pulls of multiply s+1 overlap the products of
 * multiply s.  The event must outlive the calls that use the block; NULL (default) = ordered on the ctx stream. */
int32_t mb_block_set_ready_event(mb_block* blk, void* cuda_event);
/* Breeze `.t` (no copy) and `m(r0 until r1, c0 until c1)` (a view, majorStride = parent rows),
 * as used by BlockMatrix.scala:198,213,299. */
int32_t mb_block_view_t(mb_ctx* ctx, const mb_block* blk, mb_block** out);
int32_t mb_block_slice(mb_ctx* ctx, const mb_block* blk, int32_t r0, int32_t r1, int32_t c0, int32_t c1,
                       mb_block** out);

/* ---- a1: SubMatrix.multiply (matrix/SubMatrix.scala:87-91, :107-111; inline twins
 *      matrix/DenseVecMatrix.scala:122,129,1676) -> Breeze `*` -> netlib dgemm -------------- */
/* C = A*B (accumulate=0) or C += A*B (accumulate=1; the k-way reduceByKey sum of
 * BlockMatrix.scala:177 fused into the product).  fp64: DMMA tensor-core kernel (TMA staged).
 * bf16 inputs: tcgen05 kernel with fp32 TMEM accumulation, C may be F32 or BF16. */
int32_t mb_block_gemm(mb_ctx* ctx, const mb_block* A, const mb_block* B, mb_block* C, int32_t accumulate);
/* Same GEMM on raw device pointers (column-major, BLAS trans flags 'N'/'T'). */
int32_t mb_dgemm_device(mb_ctx* ctx, char transa, char transb, int32_t m, int32_t n, int32_t k,
                        double alpha, const double* A, int32_t lda, const double* B, int32_t ldb,
                        double beta, double* C, int32_t ldc);
/* The third-party seam itself: com.github.fommil.netlib.BLAS.dgemm(transa, transb, m, n, k, alpha,
 * a, aOffset, lda, b, bOffset, ldb, beta, c, cOffset, ldc) with HOST arrays (JVM double[]).
 * Uploads, multiplies on the GPU, downloads C.  This is the end-to-end (e2e) entry bench.py times. */
int32_t mb_dgemm_host(mb_ctx* ctx, char transa, char transb, int32_t m, int32_t n, int32_t k,
                      double alpha, const double* a, int64_t a_offset, int32_t lda,
                      const double* b, int64_t b_offset, int32_t ldb,
                      double beta, double* c, int64_t c_offset, int32_t ldc);
/* fp64 arithmetic mode of the block GEMM.  MB_FP64_NATIVE (default): the DMMA kernel, true IEEE fp64 FMAs.
 * MB_FP64_INT8_SPLIT: large 'N','N' products run on the int8 tensor cores (tcgen05.mma.kind::i8) from `slices`
 * 7-bit digit planes per operand (Ozaki split; 2..8, 7 recommended): error <= ~K * 2^(-7*slices+2) relative to
 * rowmax(A) * colmax(B), i.e. well inside 1e-10 for well-scaled data but NOT an element-wise fp64 guarantee, hence
 * opt-in.  Products the split does not cover (transposed views, small blocks, K too large for exact int32
 * accumulation) silently use the native kernel. */
#define MB_FP64_NATIVE      0
#define MB_FP64_INT8_SPLIT  1   /* 7-bit digits (|d| <= 64):  P = 7*slices - 1 fractional bits, K*slices < 2^19  */
#define MB_FP64_INT8_SPLIT8 2   /* 8-bit digits (|d| <= 128): P = 8*slices - 2 fractional bits, K*slices < 2^17;
                                   slices = 5 gives 38 bits in 15 int8 GEMMs (vs 42 bits in 21 for 7-bit x 6)     */
int32_t mb_set_fp64_mode(mb_ctx* ctx, int32_t mode, int32_t slices);

/* Force the generic (non-TMA, CUDA-core DFMA) kernel: test hook + path for odd ld / unaligned views. */
int32_t mb_dgemm_device_generic(mb_ctx* ctx, char transa, char transb, int32_t m, int32_t n, int32_t k,
                                double alpha, const double* A, int32_t lda, const double* B, int32_t ldb,
                                double beta, double* C, int32_t ldc);

/* ---- a2/a10: SubMatrix.add/subtract/scalar ops (matrix/SubMatrix.scala:41-85,123-131),
 *      BlockMatrix.subtractBy/divideBy (matrix/BlockMatrix.scala:414-452) ------------------- */
int32_t mb_block_add(mb_ctx* ctx, const mb_block* A, const mb_block* B, mb_block* out);      /* A + B */
int32_t mb_block_sub(mb_ctx* ctx, const mb_block* A, const mb_block* B, mb_block* out);      /* A - B */
int32_t mb_block_hadamard(mb_ctx* ctx, const mb_block* A, const mb_block* B, mb_block* out); /* A :* B (BlockMatrix.scala:494-500) */
/* out = alpha*A + beta  (add(b): alpha=1; multiply(b): beta=0; subtractBy(b): alpha=-1, beta=b) */
int32_t mb_block_axpb(mb_ctx* ctx, const mb_block* A, double alpha, double beta, mb_block* out);
/* BDM.zeros / BDM.fill: every element of the (possibly strided) block := value */
int32_t mb_block_fill(mb_ctx* ctx, mb_block* blk, double value);
/* out = A / b  (true IEEE division, SubMatrix.divide) and out = b / A (divideBy) */
int32_t mb_block_div(mb_ctx* ctx, const mb_block* A, double b, int32_t b_over_a, mb_block* out);
/* ---- a9: BlockMatrix.transpose -> denseBlock.t.copy (matrix/BlockMatrix.scala:514-523) -- */
int32_t mb_block_transpose(mb_ctx* ctx, const mb_block* A, mb_block* out);
/* Materialise a (possibly strided / transposed) view into a packed block (Breeze `.copy`). */
int32_t mb_block_copy(mb_ctx* ctx, const mb_block* A, mb_block* out);
/* BlockMatrix.sum per block (matrix/BlockMatrix.scala:467-472) */
int32_t mb_block_sum(mb_ctx* ctx, const mb_block* A, double* sum_out);

/* ---- vector side of the path (SURVEY 8f-4): a vector is a block with one column (or one row) ----
 * y = A x (+ y): SubMatrix.multiply(v: Vector) (matrix/SubMatrix.scala:131-139) -> Breeze `BDM * BDV` -> netlib dgemv;
 * used per block by BlockMatrix.multiply(v: DistributedVector / BDV) (matrix/BlockMatrix.scala:240-274), whose
 * reduceByKey sum is `accumulate`.  A may be a transposed view (row-major rows of a DenseVecMatrix,
 * matrix/DenseVecMatrix.scala:178-191).  Reads A once: 8*rows*cols bytes. */
int32_t mb_block_gemv(mb_ctx* ctx, const mb_block* A, const mb_block* x, mb_block* y, int32_t accumulate);
/* x^T y: DistributedVector.multiply, row x column case (matrix/DistributedVector.scala:164-176) -> Breeze `v.t * w`. */
int32_t mb_block_dot(mb_ctx* ctx, const mb_block* x, const mb_block* y, double* dot_out);
/* out = x y^T: DistributedVector.multiply, column x row case (matrix/DistributedVector.scala:149-161)
 * -> Breeze `v * w.t` -> dgemm with k = 1. */
int32_t mb_block_ger(mb_ctx* ctx, const mb_block* x, const mb_block* y, mb_block* out);

/* ---- f4: the local step of DenseVecMatrix.luDecompose / choleskyDecompose / inverse
 *      (matrix/DenseVecMatrix.scala:283-466, 475-561, 568-764), which the reference hands to Breeze -> LAPACK
 *      (brzLU = dgetrf, brzCholesky = dpotrf, brzInv = dgetrf + dgetri, `\` = triangular / general solves).
 *      Recursive on the device: the flops run in the DMMA GEMM, the leaves in small panel kernels. ---- */
/* In place: unit-lower L and U packed like dgetrf; perm_out (rows entries, host, may be NULL) receives the reference's
 * permutation array: row i of L*U is row perm_out[i] of A.  A singular pivot is not an error (as with brzLU). */
int32_t mb_block_lu(mb_ctx* ctx, mb_block* A, int32_t* perm_out);
/* In place: L (lower, A = L L^T), strict upper triangle zeroed (Breeze `cholesky`); reads the lower triangle only.
 * MB_ERR_CUDA ("not positive definite") if a pivot is not positive. */
int32_t mb_block_cholesky(mb_ctx* ctx, mb_block* A);
/* out = A^-1 (partial-pivoting LU + two triangular solves of the permuted identity); MB_ERR_CUDA if exactly singular. */
int32_t mb_block_inverse(mb_ctx* ctx, const mb_block* A, mb_block* out);
/* T X = B in place (B := X), T triangular (lower / upper, unit or explicit diagonal); with transposed views of T and B
 * this also covers X T = B.  Used for `l \ b` and `b * inv(u)` of the block algorithms. */
int32_t mb_block_trsm(mb_ctx* ctx, const mb_block* T, int32_t lower, int32_t unit_diagonal, mb_block* B);

/* ---- a11: MTUtils.randomDenVecMatrix / randomBlockMatrix input generation
 *      (utils/MTUtils.scala:34-73, rdd/RandomRDD.scala:28-101, utils/RandomDataGenerator.scala:53-65,113-131).
 * Fills `count` consecutive values of partition stream `partition_seed` (one XORShift stream per
 * RDD partition), bit-exact with UniformGenerator(lo,hi).nextValue(), starting at value index
 * `first` of that stream, written into blk in the order the reference fills it
 * (row_major=1: DenseVecMatrix rows, Array.fill(cols); row_major=0: BDM.create column-major). */
int32_t mb_fill_uniform(mb_ctx* ctx, mb_block* blk, int64_t partition_seed, int64_t first,
                        double lo, double hi, int32_t row_major);
/* Host-side pieces of the same generator (pure integer logic, exported for the host mirror):
 * MTUtils.hashSeed (MurmurHash3.bytesHash over a 64-byte buffer) and the per-partition seeds
 * = successive java.util.Random(seed).nextLong() (rdd/RandomRDD.scala:28-45). */
int64_t mb_hash_seed(int64_t seed);
int32_t mb_partition_seeds(int64_t seed, int32_t num_partitions, int64_t* seeds_out);

/* ---- a7/a8: strategy + partitioning (pure integer logic) --------------------------------- */
/* MTUtils.splitMethod(m,k,n,cores) (utils/MTUtils.scala:150-175, dimToSplit :204-213) */
int32_t mb_choose_split(int64_t m, int64_t k, int64_t n, int32_t cores, int32_t out_mkn[3]);
/* DenseVecMatrix.multiply(other,cores,broadcastThreshold) chooser (matrix/DenseVecMatrix.scala:196-231,
 * matrix/BlockMatrix.scala:87-122).  other_is_block selects the `case that: BlockMatrix` arm.
 * Returns strategy in *strategy: 0 = broadcast B (this.multiply(that.toBreeze())),
 * 1 = broadcast A (the reference's quirk arm), 2 = shuffle with out_mkn. */
int32_t mb_choose_strategy(int64_t a_rows, int64_t a_cols, int64_t b_cols, int32_t cores,
                           int32_t broadcast_threshold_mb, int32_t other_is_block,
                           int32_t* strategy, int32_t out_mkn[3]);
/* MatrixMultPartitioner (rdd/MatrixMultPartitioner.scala:12-22) with the seq formula of
 * matrix/BlockMatrix.scala:163,168: seq = i*n*k + j*k + kk. */
int32_t mb_mult_partition(int32_t i, int32_t j, int32_t kk, int32_t m, int32_t k, int32_t n);
/* MatrixElemOpPartitioner (rdd/MatrixElemOpPartitioner.scala:16) */
int32_t mb_elem_partition(int32_t row, int32_t col, int32_t blks_by_col);
/* ceil-based block sizing (matrix/BlockMatrix.scala:73-74, matrix/DenseVecMatrix.scala:1091-1094):
 * block length = ceil(total/parts); actual number of blocks = ceil(total/block_len). */
int32_t mb_block_len(int64_t total, int32_t parts, int32_t* block_len, int32_t* actual_parts);

/* ---- a3/a4: BlockMatrix.multiply(other: BlockMatrix) on ONE device
 *      (matrix/BlockMatrix.scala:149-186): all m*k*n block products in seq order, the k partials of
 *      each C tile accumulated in place.  A_tiles[i*k+kk], B_tiles[kk*n+j], C_tiles[i*n+j]
 *      (MatrixElemOpPartitioner order).  Multi-GPU sharding of the seq list is done by the host
 *      (marlin_b200.matrix.BlockMatrix) with one process per GPU. */
int32_t mb_matmul_blocked(mb_ctx* ctx, mb_block* const* A_tiles, mb_block* const* B_tiles,
                          int32_t m, int32_t k, int32_t n, mb_block* const* C_tiles);
/* The share of that multiply one rank runs: only the C blocks listed in c_ids (c = i*n + j), each with its full
 * kk-sum.  Tile slots this rank does not need may be NULL.  fp64 'N' blocks run as ONE persistent grouped launch
 * (K loop concatenated over kk, no C read-modify-write); anything else falls back to per-product launches. */
int32_t mb_matmul_blocked_subset(mb_ctx* ctx, mb_block* const* A_tiles, mb_block* const* B_tiles,
                                 int32_t m, int32_t k, int32_t n, mb_block* const* C_tiles,
                                 const int32_t* c_ids, int32_t num_c);

/* The same multiply for JVM-held blocks (HOST column-major fp64 arrays in, host arrays out): the entry a
 * `BlockMatrix.multiply` whose SubMatrix data still lives on the heap would bind.  A_host[i*k+kk] is the packed
 * (row_len[i] x k_len[kk]) tile, B_host[kk*n+j] the (k_len[kk] x col_len[j]) tile, C_host[i*n+j] receives the
 * (row_len[i] x col_len[j]) result.  Uploads, the m*k*n DMMA products (seq order, kk accumulated in the epilogue)
 * and downloads are pipelined on separate streams: tiles are uploaded in first-use order and every C tile
 * starts its D2H as soon as its last partial is done.  Pinned host memory gives full PCIe overlap; pageable
 * memory still works (the copies just serialise).  This is the end-to-end path bench.py times at N=1. */
int32_t mb_matmul_blocked_host(mb_ctx* ctx, const double* const* A_host, const double* const* B_host,
                               int32_t m, int32_t k, int32_t n, const int32_t* row_len, const int32_t* k_len,
                               const int32_t* col_len, double* const* C_host);

/* a5: DenseVecMatrix.multiply(B: BDM[Double]) (matrix/DenseVecMatrix.scala:1660-1680) for the row shard one process
 * holds: C_rows = A_rows * B.  A_rows / C_rows are row-major shards (transposed views of the column-major array
 * underneath), B is the broadcast matrix; the rows never change GPU, so N ranks run N independent calls. */
int32_t mb_matmul_rowsharded(mb_ctx* ctx, const mb_block* A_rows, const mb_block* B, mb_block* C_rows);
/* The same for JVM-held rows: A_host = the shard's rows back to back (row-major, k doubles per row: the packed
 * `rowsMat` of :1672-1675), B_host = column-major k x n, C_host receives rows x n row-major.  Row chunks of ~256 MiB
 * are pipelined over three streams (H2D of chunk c+1, the DMMA product of chunk c, D2H of chunk c-1). */
int32_t mb_matmul_rowsharded_host(mb_ctx* ctx, const double* A_host, int64_t rows, int32_t k, const double* B_host,
                                  int32_t n, double* C_host);

/* ---- peer memory: NVLink P2P between the per-GPU processes of one box (CUDA IPC) ------------------------------
 * Replaces the shuffle transport of the multiply (matrix/BlockMatrix.scala:161-177): a rank maps the tile buffers
 * of the others once, pulls the tiles it needs with copy-engine DMA (mb_memcpy_async on a side stream) and lets its
 * GEMM epilogue store partial products directly into the reducing rank's memory (pass a peer pointer as C).
 * Ordering between processes uses stream-ordered flags (monotonic epochs) living in exported device memory. */
int32_t mb_ipc_export(mb_ctx* ctx, const void* device_ptr, uint8_t handle_out[64], int64_t* offset_out,
                      int64_t* alloc_bytes_out);
int32_t mb_ipc_open(mb_ctx* ctx, const uint8_t handle[64], void** base_out);     /* cached per handle */
int32_t mb_ipc_close_all(mb_ctx* ctx);
int32_t mb_flags_alloc(mb_ctx* ctx, int32_t count, void** flags_out);            /* zeroed uint64[count], cudaMalloc'd */
int32_t mb_flags_free(mb_ctx* ctx, void* flags);
int32_t mb_flag_signal(mb_ctx* ctx, void* flag, int64_t value);   /* on the ctx stream: release-store (system scope) */
int32_t mb_flag_wait(mb_ctx* ctx, const void* flag, int64_t value); /* on the ctx stream: wait until *flag >= value */
int32_t mb_memcpy_async(mb_ctx* ctx, void* dst, const void* src, int64_t bytes);   /* D2D (local or peer) on the ctx stream */

/* ---- (e) BlockMatrix.multiply across the GPUs of one box, entirely behind this ABI ---------------------------------
 * One process (or thread with its own ctx) per GPU.  mb_comm is the analogue of the executors of one SparkContext:
 * created once, collectively, by `world` ranks that pass the same `session` string (unique per communicator: it names a
 * POSIX shared-memory segment used for rendezvous and per-call tile directories — no network, no torch, no MPI).
 * mb_matmul_blocked_dist is the whole of matrix/BlockMatrix.scala:159-178 — MatrixMultPartitioner mapping
 * (seq = i*n*k + j*k + kk dealt to ranks in contiguous ranges: mb_dist_plan), tile replication (NVLink peer-memory
 * pulls overlapped with the products), the m*k*n DMMA block products (one persistent launch per rank; two where a k
 * partial crosses GPUs) and the reduceByKey of the k partials (reduce-scatter by the GEMM epilogues between two holders,
 * staged adds otherwise).
 * Every rank calls it with the same m, k, n, lengths and owner maps; A_tiles[i*k+kk] / B_tiles[kk*n+j] are non-NULL
 * exactly where the owner map names this rank; C_tiles[i*n+j] must be a preallocated (row_len[i] x col_len[j]) block
 * (F64, or F32 for BF16 inputs) wherever mb_dist_plan's c_owner names this rank, and receives the finished tile there.
 * Asynchronous like every other compute entry: ordered on the ctx stream.  Flags between the processes are stream memory
 * operations and peer stores, never kernels (nothing the resident GEMM waits for needs an SM); in-kernel waits are bounded
 * by MARLIN_B200_TIMEOUT_S, host-side waits too (then the communicator aborts itself and the call returns MB_ERR_TIMEOUT).
 * Give every stream its own hardware queue: CUDA_DEVICE_MAX_CONNECTIONS=32 before the CUDA context is created. */
typedef struct mb_comm mb_comm;
#define MB_ERR_TIMEOUT       -7   /* a peer did not answer within MARLIN_B200_TIMEOUT_S (default 120 s) -> RuntimeException */
int32_t mb_comm_init(mb_ctx* ctx, int32_t rank, int32_t world, const char* session, mb_comm** out);
int32_t mb_comm_destroy(mb_comm* comm);
int32_t mb_comm_rank(const mb_comm* comm);
int32_t mb_comm_world(const mb_comm* comm);
int32_t mb_comm_barrier(mb_comm* comm);            /* host-side barrier of the ranks */
int32_t mb_comm_abort(mb_comm* comm);              /* release every wait queued on this rank (results garbage); the comm is dead */
int32_t mb_comm_check(mb_comm* comm);              /* MB_ERR_TIMEOUT if a device-side wait for a peer ever gave up */
/* MatrixMultPartitioner + placement: product seq -> rank (m*k*n entries) and C tile -> owning rank (m*n entries). */
int32_t mb_dist_plan(int32_t m, int32_t k, int32_t n, int32_t world, int32_t* product_rank_out, int32_t* c_owner_out);
int32_t mb_matmul_blocked_dist(mb_comm* comm, mb_block* const* A_tiles, const int32_t* a_owner,
                               mb_block* const* B_tiles, const int32_t* b_owner, int32_t m, int32_t k, int32_t n,
                               const int32_t* row_len, const int32_t* k_len, const int32_t* col_len, int32_t dtype,
                               mb_block* const* C_tiles);

/* The same multiply END TO END with HOST tiles (what bench.py reports as e2e at N > 1): every input tile is uploaded by
 * ONE of the ranks that need it (a_home / b_home; mb_dist_host_homes spreads them over the PCIe links) and pulled over
 * NVLink by the others, band by band; one grouped DMMA launch per rank starts on the first bands; the two holders of a
 * k-split C tile each reduce and download a checkerboard of its sub-blocks, hidden behind the rest of the GEMM.
 * A_host / B_host: packed column-major tiles, non-NULL where homed; C_host[i*n+j]: the packed host tile, non-NULL on
 * every rank that computes a partial of it (use one mb_host_alloc_shared array per tile so that the ranks fill one copy).
 * fp64, at most two holders per C tile.  Blocking. */
int32_t mb_dist_host_homes(int32_t m, int32_t k, int32_t n, int32_t world, int32_t* a_home, int32_t* b_home);
int32_t mb_matmul_blocked_dist_host(mb_comm* comm, const double* const* A_host, const int32_t* a_home,
                                    const double* const* B_host, const int32_t* b_home, int32_t m, int32_t k, int32_t n,
                                    const int32_t* row_len, const int32_t* k_len, const int32_t* col_len,
                                    double* const* C_host);
/* Pinned host memory shared by the processes of one box (POSIX shm `name` + cudaHostRegister). */
int32_t mb_host_alloc_shared(const char* name, int64_t bytes, void** out);
int32_t mb_host_free_shared(const char* name, void* ptr, int64_t bytes, int32_t unlink_name);

/* ---- sparse blocks: `new SubMatrix(spMatrix = ...)` (matrix/SubMatrix.scala:22-25) holding a SparseMatrix
 *      (matrix/Matrices.scala:136-253).  An mb_spblock is CSC on the device, the reference's one SparseVector per column:
 *      col_ptr int32[cols+1] (col_ptr[0] = 0, non-decreasing; an empty column has col_ptr[c] == col_ptr[c+1]),
 *      row_idx int32[nnz] strictly increasing within each column and inside [0, rows), val fp64[nnz].
 *      The products write a dense column-major result (a dense mb_block, any view), as the reference does.  Each output
 *      element is a sequential sum from +0.0 in the reference's order with one rounded multiply and one rounded add per
 *      term (the JVM never fuses them); accumulate = 1 adds the finished sum to C with one rounding, i.e. exactly
 *      mb_block_add of a separate product (the k-way reduceByKey of matrix/BlockMatrix.scala:177). ---- */
typedef struct mb_spblock mb_spblock;
/* The validation mb_spblock_upload runs before anything is uploaded (pure host logic): MB_ERR_INVALID_ARG for a
 * col_ptr that does not start at 0 or decreases, or a row index out of range or not strictly increasing in its column. */
int32_t mb_csc_check(int32_t rows, int32_t cols, const int32_t* col_ptr, const int32_t* row_idx);
int32_t mb_spblock_upload(mb_ctx* ctx, int32_t rows, int32_t cols, const int32_t* col_ptr, const int32_t* row_idx,
                          const double* val, mb_spblock** out);
/* host arrays of cols+1, nnz and nnz entries */
int32_t mb_spblock_download(mb_ctx* ctx, const mb_spblock* sp, int32_t* col_ptr, int32_t* row_idx, double* val);
int32_t mb_spblock_info(const mb_spblock* sp, int32_t* rows, int32_t* cols, int64_t* nnz);
int32_t mb_spblock_free(mb_ctx* ctx, mb_spblock* sp);
/* A new block with the same structure and values (the scalar ops of SubMatrix.scala:52-58,71-85,121-129 map a copy). */
int32_t mb_spblock_copy(mb_ctx* ctx, const mb_spblock* sp, mb_spblock** out);
/* The stored values as a non-owning (nnz x 1) fp64 mb_block, so mb_block_axpb / mb_block_div map them in place:
 * the scalar ops touch the stored values only (A + 1 leaves implicit zeros at zero). */
int32_t mb_spblock_values(mb_ctx* ctx, mb_spblock* sp, mb_block** out);
/* SparseMatrix.toDense (matrix/Matrices.scala:106-119): out (rows x cols fp64, any view) := the dense matrix. */
int32_t mb_spblock_to_dense(mb_ctx* ctx, const mb_spblock* sp, mb_block* out);
/* SparseMatrix.rand(rows, cols, sparsity) (matrix/Matrices.scala:157-173): every column holds exactly
 * count = (int)(cols * sparsity) distinct rows (the count follows numCols, as in the reference), sorted, values U[0,1).
 * The reference draws from an unseeded java.util.Random; here column c of a block seeded with `partition_seed` (one of
 * mb_partition_seeds, as dense blocks are seeded) has its own splitmix64 stream, rows are chosen by selection sampling,
 * so a seed reproduces the matrix.  Generated on the device.  mb_sparse_rand_count is the count and its checks:
 * MB_ERR_INVALID_ARG for a negative or NaN sparsity, a count above rows (where the reference loops forever) or
 * count * cols >= 2^31 (matrix/Matrices.scala:71). */
int32_t mb_sparse_rand_count(int32_t rows, int32_t cols, double sparsity, int32_t* count);
int32_t mb_spblock_rand(mb_ctx* ctx, int32_t rows, int32_t cols, double sparsity, int64_t partition_seed, mb_spblock** out);
/* SubMatrix.multiply, (dense, sparse) arm (SubMatrix.scala:95-97) -> LibMatrixMult.multDenseSparse
 * (matrix/LibMatrixMult.scala:15-41): C(r,j) = sum over B's column j in stored order of B(k,j)*A(r,k); a column holding
 * exactly one entry equal to 1.0 copies A's column (:28-29).  MB_ERR_DIM_MISMATCH "matrix dimension mismatch: a v.s b". */
int32_t mb_spmm_dense_sparse(mb_ctx* ctx, const mb_block* A, const mb_spblock* B, mb_block* C, int32_t accumulate);
/* SubMatrix.multiply, (sparse, dense) arms (SubMatrix.scala:98-100,112-114) -> LibMatrixMult.multSparseDense
 * (matrix/LibMatrixMult.scala:43-77) AS DEFINED: C(r,j) = sum over k ascending of A(r,k)*B(k,j) over the stored A(r,k).
 * The reference's loop indexes B with `i * cd + bi` (:60) and is only right for K <= 32 and N <= 32 (DESIGN.md,
 * documented deviations); B's offset / ld / transpose are honoured as mb_block_gemm honours them. */
int32_t mb_spmm_sparse_dense(mb_ctx* ctx, const mb_spblock* A, const mb_block* B, mb_block* C, int32_t accumulate);
/* SubMatrix.multiply, (sparse, sparse) arm (SubMatrix.scala:92-94) -> SparseMatrix.multiply (matrix/Matrices.scala:122-152):
 * C(r,j) = sum over B's column j in stored order of B(k,j)*A(r,k), over the stored A(r,k). */
int32_t mb_spgemm_to_dense(mb_ctx* ctx, const mb_spblock* A, const mb_spblock* B, mb_block* C, int32_t accumulate);

/* ---- rows <-> blocks on device (matrix/DenseVecMatrix.scala:1084-1223, 1259-1328;
 *      matrix/BlockMatrix.scala:575-594): a DenseVecMatrix shard is a row-major (rows x cols)
 *      buffer, i.e. a transposed block; these are strided copies (mb_block_copy on views). */

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* MARLIN_B200_H */
