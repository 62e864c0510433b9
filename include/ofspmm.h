/*
 * ofspmm.h — C ABI of the B200-native SpMM operator library (libofspmm_b200.so).
 *
 * This is the drop-in boundary for the OneFlow user op `spmm_csr` (+ `spmm_csr_grad_b`,
 * `sddmm_csr`): the body of `user_op::OpKernel::Compute(KernelComputeContext*)`
 * (reference: oneflow/core/framework/op_kernel.h:305-308) pulls raw pointers, shapes, attrs and
 * the `cudaStream_t` out of `ctx` and calls the functions below (glue sources:
 * of-spmm_b200/oneflow_glue/, binding walk-through: INTEGRATION.md).
 *
 * Conventions — each mirrors a rule of the reference's kernel contract (SURVEY.md §8b):
 *   - plain pointers and sizes only; every data pointer is a DEVICE pointer unless the name ends
 *     in `_host`; no torch / OneFlow types;
 *   - nothing here allocates or frees device memory and nothing synchronises the stream or the
 *     device: temporary storage is a caller-owned workspace sized by the matching
 *     `*_workspace_bytes()` query, which plays the role of `SetInferTmpSizeFn`
 *     (oneflow/core/framework/user_op_kernel_registry.h:60,90;
 *      oneflow/user/kernels/unsorted_segment_sum_kernel.cpp:191-202);
 *   - work is enqueued on the given stream and the call returns (async contract of
 *     oneflow/core/framework/op_kernel.h:311); all calls are CUDA-graph capturable
 *     (user_op::CudaGraphSupport, oneflow/core/kernel/cuda_graph_support.h:28-42);
 *   - no global mutable state, no cudaSetDevice: the library is re-entrant and runs on whatever
 *     device is current on the calling thread (oneflow/core/vm/virtual_machine.cpp:69-77);
 *   - errors are int status codes; no C++ exception crosses the boundary.  The glue turns a
 *     non-zero status into CHECK / LOG(FATAL) like OF_CUDA_CHECK does
 *     (oneflow/core/device/cuda_util.h:54-57);
 *   - outputs are fully overwritten (the framework does not zero them,
 *     oneflow/core/vm/op_call_instruction_policy.cpp:78-85);
 *   - column indices outside [0, cols) are skipped, as the reference's segment-sum skips
 *     out-of-range ids (oneflow/user/kernels/unsorted_segment_sum_kernel_util.cpp:35-39): nothing
 *     is loaded for such an entry, in every product and in the transpose (where they end up behind
 *     the last row of A^T with column -1).
 *
 * dtype codes reuse OneFlow's DataType numbering (oneflow/core/common/data_type.proto:4-17) so
 * the glue passes `tensor->data_type()` through unchanged.
 */
#ifndef OFSPMM_H_
#define OFSPMM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define OFSPMM_API
#else
#define OFSPMM_API __attribute__((visibility("default")))
#endif

/* Same object as cudaStream_t (CUstream_st*); spelled out so C callers need no CUDA headers. */
typedef struct CUstream_st* ofspmm_stream_t;

/* oneflow::DataType values (data_type.proto:4-17). */
enum {
  OFSPMM_DTYPE_FLOAT = 2,     /* kFloat    */
  OFSPMM_DTYPE_INT32 = 5,     /* kInt32    */
  OFSPMM_DTYPE_INT64 = 6,     /* kInt64    */
  OFSPMM_DTYPE_BFLOAT16 = 11  /* kBFloat16 */
};

/* Value dtype of a PATTERN matrix: every stored entry has value 1.0 and nothing is stored, so
 * `val` must be NULL (a non-NULL `val` returns OFSPMM_ERR_INVALID_ARG: a forgotten dtype field is
 * caught, not ignored).  The code lies outside OneFlow's DataType numbering on purpose: no tensor
 * dtype means "no tensor".  Combines with both dense dtypes; the CSR stream per non-zero drops
 * from idx+val bytes to idx bytes. */
enum { OFSPMM_VAL_UNIT = 0x100 };

enum {
  OFSPMM_OK = 0,
  OFSPMM_ERR_INVALID_ARG = 1,       /* null pointer, negative size, inconsistent shape        */
  OFSPMM_ERR_UNSUPPORTED_DTYPE = 2, /* dtype combination without a kernel                      */
  OFSPMM_ERR_WORKSPACE = 3,         /* workspace null / misaligned / smaller than the query    */
  OFSPMM_ERR_CUDA = 4,              /* a CUDA runtime call or launch failed (cudaGetLastError) */
  OFSPMM_ERR_TOO_LARGE = 5,         /* rows >= 2^31-1, or nnz >= 2^31-1 with int32 indices      */
  OFSPMM_ERR_NO_DEVICE = 6          /* no sm_100 device current on this thread                 */
};

/* A (rows × cols) in CSR.  crow has rows+1 entries, col / val have nnz entries.
 * idx_dtype ∈ {INT32, INT64} applies to both crow and col (INDEX_DATA_TYPE_SEQ,
 * oneflow/core/common/data_type_seq.h:50-52).  val_dtype ∈ {FLOAT, BFLOAT16, VAL_UNIT}; BFLOAT16
 * values are only accepted together with a BFLOAT16 dense operand; VAL_UNIT (pattern matrix, val
 * NULL) is accepted by the forward entry points, ofspmm_bwd_b (A and At), the transient and
 * cached backward, the transpose and ofspmm_fwd_host, not by the SDDMM.  `val` may be NULL for
 * ofspmm_sddmm.
 * Ranges: rows < 2^31-1 for both index dtypes; nnz < 2^31-1 with INT32 indices, while INT64
 * indices take any nnz whose (rows + nnz) / 256 merge-path tasks stay below 2^30
 * (nnz below about 2.7e11). */
typedef struct ofspmm_csr {
  int64_t rows;
  int64_t cols;
  int64_t nnz;
  const void* crow;
  const void* col;
  const void* val;
  int32_t idx_dtype;
  int32_t val_dtype;
} ofspmm_csr;

/* ---- Per-call options of the *_ex entry points.  Zero-initialise for the defaults; a NULL
 * `opts` means all defaults.  Everything a launch depends on is in the arguments: the library
 * reads no environment variable and keeps no mutable global (SURVEY.md §8b "Threading"). */
enum {
  OFSPMM_FWD_ACCUMULATE = 1, /* C += A·B instead of C = A·B (second pass of a column-bucketed product) */
  OFSPMM_FWD_BIAS = 2,       /* fused epilogue: + bias[j] (opts->bias: n elements of the dense dtype)    */
  OFSPMM_FWD_RELU = 4,       /* fused epilogue: max(., 0), after the bias (GCNConv; precedent for a
                                fused epilogue: oneflow/user/kernels/cublas_fused_mlp_kernel.cu)        */
  OFSPMM_ORDER_DYNAMIC = 8,  /* persistent grid draws its tasks from a counter, in launch order         */
  OFSPMM_ORDER_STATIC = 16,  /* persistent grid uses the fixed interleave (warp w: tasks w, w+W, ...)   */
  /* bf16 products computed in several passes (column buckets): the running row sums stay in the
   * fp32 buffer opts->acc32 (rows x n, packed) between the passes, so the result is rounded to
   * bf16 once.  first pass: ACC32_OUT; middle: IN | OUT; last: IN (+ epilogue) -> C.             */
  OFSPMM_FWD_ACC32_IN = 32,
  OFSPMM_FWD_ACC32_OUT = 64,
  /* mean aggregation (torch.sparse.mm(reduce="mean")): each row's complete fp32 sum is divided by
   * the row's stored-entry count crow[i+1] - crow[i], before the bias and the ReLU.  Weighted and
   * pattern matrices alike.  An empty row gives 0 (then bias / ReLU).  Entries with a column
   * outside [0, cols) add nothing but still count in the divisor.  Cannot be combined with
   * ACCUMULATE or ACC32_IN / ACC32_OUT (OFSPMM_ERR_INVALID_ARG): the division applies to this
   * call's complete row sum only. */
  OFSPMM_FWD_MEAN = 128
};
/* Task order when neither ORDER bit is set (measured default, see DESIGN.md §3.2). */
#ifndef OFSPMM_DEFAULT_DYNAMIC_ORDER
#define OFSPMM_DEFAULT_DYNAMIC_ORDER 1
#endif

/* Kernel variant of the forward-shaped products.  AUTO decides from (rows, nnz, n, dtype); with the
 * row-length histogram on the host, ofspmm_choose_variant() returns an EXPLICIT code. */
enum {
  OFSPMM_VARIANT_AUTO = 0,
  OFSPMM_VARIANT_ITEMS64 = 1,  /* 64 merge items per warp task (small problems: 4x more warps)      */
  OFSPMM_VARIANT_ROWPAR = 2,   /* sub-warp per row instead of nnz-parallel groups (short rows x
                                  narrow dense operand)                                              */
  OFSPMM_VARIANT_ROWS = 4,     /* whole rows per lane group, ONE launch, no partition / carries /
                                  fix-up: small problems whose longest row is short (needs int32
                                  indices and 16-byte dense rows of <= 512 bytes, else ITEMS64)      */
  OFSPMM_VARIANT_EXPLICIT = 0x100
};

typedef struct ofspmm_opts {
  uint32_t flags;         /* OFSPMM_FWD_* | OFSPMM_ORDER_*                                           */
  int32_t tasks_per_warp; /* 0: persistent grid.  k > 0: CTAs retire after ~k tasks per warp, so a
                             kernel on another stream (a collective, the peer pull) gets SMs while
                             this one runs                                                          */
  int32_t variant;        /* OFSPMM_VARIANT_AUTO or a code from ofspmm_choose_variant               */
  int32_t reserve_ctas_per_sm; /* persistent grid of (occupancy - r) CTAs per SM: every SM keeps r CTA
                             slots (128 threads, <= 64 registers each) free for the 128-thread
                             exchange kernels that overlap this product (pull / combine / signal)   */
  const void* plan;       /* device plan from ofspmm_plan_build for THIS (crow, variant); NULL: the
                             partition is recomputed inside the call                                */
  size_t plan_bytes;
  const void* bias;       /* OFSPMM_FWD_BIAS: n elements of the dense dtype                          */
  void* acc32;            /* OFSPMM_FWD_ACC32_*: rows x n fp32, 16-byte aligned                      */
} ofspmm_opts;

/* ---- SpMM forward: C[rows × n] = A · B[cols × n]  (replaces the `spmm_csr` kernel body; data
 * movement analogue in the reference: GatherForwardGpu + UnsortedSegmentRowSumGpu,
 * oneflow/user/kernels/gather_kernel_util.cu:28-41,
 * oneflow/user/kernels/unsorted_segment_sum_kernel_util.cu:96-117).
 * B and C are row-major, contiguous, of `dense_dtype` ∈ {FLOAT, BFLOAT16}; accumulation is fp32,
 * bf16 outputs are rounded once.  Deterministic: the summation order depends only on
 * (crow, n, dtype), never on scheduling. */
OFSPMM_API size_t ofspmm_fwd_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int64_t n,
                                             int dense_dtype);
OFSPMM_API int ofspmm_fwd(const ofspmm_csr* A, const void* B, void* C, int64_t n, int dense_dtype,
                          void* workspace, size_t workspace_bytes, ofspmm_stream_t stream);
/* Same with explicit row strides (in elements, >= n): B is cols × n inside a row-major buffer of
 * leading dimension ldb, C likewise with ldc — a column slice of a wider matrix, as
 * `user_op::Tensor::stride()` describes it (oneflow/core/framework/user_op_tensor.h:31-72).  Used
 * by the multi-GPU path to compute / write one column panel of the dense operands at a time
 * while the next panel's all-gather is in flight.  Workspace = ofspmm_fwd_workspace_bytes(n). */
OFSPMM_API int ofspmm_fwd_strided(const ofspmm_csr* A, const void* B, int64_t ldb, void* C,
                                  int64_t ldc, int64_t n, int dense_dtype, void* workspace,
                                  size_t workspace_bytes, ofspmm_stream_t stream);

/* Forward with options: strides as in ofspmm_fwd_strided, plus variant / plan / launch policy /
 * fused epilogue.  Workspace = ofspmm_fwd_ex_workspace_bytes(..., opts->variant). */
OFSPMM_API size_t ofspmm_fwd_ex_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int64_t n,
                                                int dense_dtype, int variant);
OFSPMM_API int ofspmm_fwd_ex(const ofspmm_csr* A, const void* B, int64_t ldb, void* C, int64_t ldc,
                             int64_t n, int dense_dtype, const ofspmm_opts* opts, void* workspace,
                             size_t workspace_bytes, ofspmm_stream_t stream);

/* ---- Plan: the task partition of one (crow, variant), computed once and kept by the caller in
 * the op's OpKernelState (oneflow/user/kernels/stateful_opkernel.cpp:919-928) for as long as `crow`
 * is unchanged; every product then skips the partition kernel.  Device buffer of
 * ofspmm_plan_bytes(), 16-byte aligned, read-only to the products (safe to share between streams). */
OFSPMM_API size_t ofspmm_plan_bytes(int64_t rows, int64_t nnz, int64_t n, int dense_dtype, int variant);
OFSPMM_API int ofspmm_plan_build(const void* crow, int idx_dtype, int64_t rows, int64_t nnz, int64_t n,
                                 int dense_dtype, int variant, void* plan, size_t plan_bytes,
                                 ofspmm_stream_t stream);

/* ---- Variant choice from the row-length histogram (north_star (2)).  `hist32_host` = the 32
 * counters of ofspmm_row_hist copied to the HOST (once, when the op state is built — never inside a
 * captured call); NULL gives the AUTO decision.  Pure host function, no CUDA call.  Rules (measured,
 * profiles/r2_variant_sweeps.md, profiles/r2_results_1gpu.md):
 *   - small problem (fewer 256-item tasks than resident warps): ROWS when no row has >= 512
 *     non-zeros, the dense rows are 16-byte vectors of <= 512 bytes and one lane group per row
 *     gives >= 8 warps per SM; otherwise ITEMS64;
 *   - else ROWPAR when the lane layout is sub-warp (dense row <= 256 bytes) and the median row,
 *     empty rows included, has fewer than 16 non-zeros;
 *   - else the base family (256-item tasks, nnz-parallel lane groups). */
OFSPMM_API int ofspmm_choose_variant(const int64_t* hist32_host, int64_t rows, int64_t nnz, int64_t n,
                                     int dense_dtype);

/* ---- Backward wrt the dense operand: dB[cols × n] = A^T · dY[rows × n]  (replaces
 * `spmm_csr_grad_b`; reference analogue = memset + atomic scatter-add,
 * oneflow/user/kernels/unsorted_segment_sum_kernel.cpp:91-117,
 * oneflow/user/kernels/embedding_kernel_util.cu:50-64).
 * Two routes:
 *   (1) `At` != NULL: a CSR of A^T built once by ofspmm_csr_transpose and kept in the op's
 *       OpKernelState; runs the forward kernel on it — deterministic, no atomics;
 *   (2) `At` == NULL: vector-atomic scatter (red.global.add.v4.f32) into an fp32 accumulator
 *       (dB itself for FLOAT, the workspace for BFLOAT16) — order-nondeterministic like the
 *       reference's cuda::atomic::Add path. */
OFSPMM_API size_t ofspmm_bwd_b_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int64_t n,
                                               int dense_dtype, int have_transpose);
OFSPMM_API int ofspmm_bwd_b(const ofspmm_csr* A, const ofspmm_csr* At, const void* dY, void* dB,
                            int64_t n, int dense_dtype, void* workspace, size_t workspace_bytes,
                            ofspmm_stream_t stream);

/* Route (3), for callers without an op state: build A^T transiently inside the workspace (stable
 * radix sort, ~5 ms for 115 M non-zeros on B200) and run the forward kernel on it — deterministic,
 * and still faster than route (2).  Workspace = ofspmm_bwd_b_transient_workspace_bytes(...)
 * (about nnz*(idx+val) + transpose scratch + the forward workspace; no value bytes for VAL_UNIT). */
OFSPMM_API size_t ofspmm_bwd_b_transient_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz,
                                                         int64_t n, int dense_dtype, int idx_dtype,
                                                         int val_dtype);
OFSPMM_API int ofspmm_bwd_b_transient(const ofspmm_csr* A, const void* dY, void* dB, int64_t n,
                                      int dense_dtype, void* workspace, size_t workspace_bytes,
                                      ofspmm_stream_t stream);

/* Route (1'), the one the OneFlow glue uses: the caller caches only the STRUCTURE of A^T
 * (t_crow[cols+1], t_col[nnz], t_perm[nnz] from ofspmm_csr_transpose — ordinary tensors owned by
 * the framework) and the values are re-gathered from A->val through t_perm on every call, so
 * in-place updates of a_val are always seen and no hidden pointer-keyed cache exists.  A pattern
 * matrix (VAL_UNIT) gathers nothing and its workspace holds no value array. */
OFSPMM_API size_t ofspmm_bwd_b_cached_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz,
                                                      int64_t n, int dense_dtype, int val_dtype);
OFSPMM_API int ofspmm_bwd_b_cached(const ofspmm_csr* A, const void* t_crow, const void* t_col,
                                   const void* t_perm, const void* dY, void* dB, int64_t n,
                                   int dense_dtype, const ofspmm_opts* opts, void* workspace,
                                   size_t workspace_bytes, ofspmm_stream_t stream);

/* out[q] = val[perm[q]]: the values of A^T from the values of A (perm = t_perm of
 * ofspmm_csr_transpose).  What ofspmm_bwd_b_cached runs internally; exported for callers that can
 * prove the values unchanged between calls (e.g. a tensor version counter) and keep t_val. */
OFSPMM_API int ofspmm_permute_values(const void* val, int val_dtype, const void* perm, int idx_dtype,
                                     int64_t nnz, void* out, ofspmm_stream_t stream);

/* ---- SDDMM value gradient: dval[p] = <dY[i,:], B[col[p],:]> for every stored entry p of row i
 * (replaces `sddmm_csr`; no reference analogue, SURVEY.md §8a5).  dval has `val_dtype` of A
 * (FLOAT, or BFLOAT16 with a BFLOAT16 dense operand); A->val is not read.  VAL_UNIT returns
 * OFSPMM_ERR_UNSUPPORTED_DTYPE: a pattern matrix has no values to differentiate. */
OFSPMM_API size_t ofspmm_sddmm_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int64_t n,
                                               int dense_dtype);
OFSPMM_API int ofspmm_sddmm(const ofspmm_csr* A, const void* dY, const void* B, void* dval,
                            int64_t n, int dense_dtype, void* workspace, size_t workspace_bytes,
                            ofspmm_stream_t stream);

OFSPMM_API int ofspmm_sddmm_ex(const ofspmm_csr* A, const void* dY, const void* B, void* dval,
                               int64_t n, int dense_dtype, const ofspmm_opts* opts, void* workspace,
                               size_t workspace_bytes, ofspmm_stream_t stream);

/* ---- Merge-path / nnz-balanced partitioner (SURVEY.md §8a6).  Splits the merged list of
 * (row-end, non-zero) items into `parts` equal spans; writes parts+1 split points
 * (out_row[k], out_nz[k]) with out_row[k] + out_nz[k] = min(k·ceil((rows+nnz)/parts), rows+nnz).
 * Device version (outputs are device int64 arrays) and its host twin (all pointers host) must
 * agree bit-for-bit; contrast the reference's equal-count BalancedSplitter
 * (oneflow/core/common/balanced_splitter.cpp:20-39). */
OFSPMM_API int ofspmm_partition(const void* crow, int idx_dtype, int64_t rows, int64_t nnz,
                                int64_t parts, int64_t* out_row, int64_t* out_nz,
                                ofspmm_stream_t stream);
OFSPMM_API int ofspmm_partition_host(const void* crow_host, int idx_dtype, int64_t rows,
                                     int64_t nnz, int64_t parts, int64_t* out_row_host,
                                     int64_t* out_nz_host);

/* ---- Row-length histogram in log2 buckets: hist[0] = empty rows, hist[b] = rows with
 * 2^(b-1) <= len < 2^b (b = 1..31).  32 device int64 counters, overwritten.  Copied to the host
 * once (op-state construction) it feeds ofspmm_choose_variant (SURVEY.md §8a6). */
OFSPMM_API int ofspmm_row_hist(const void* crow, int idx_dtype, int64_t rows, int64_t* hist32,
                               ofspmm_stream_t stream);

/* ---- Device CSR → CSR-of-A^T (stable: entries of one column keep ascending row order), the
 * one-off the op's OpKernelState runs for route (1) of ofspmm_bwd_b.  Output arrays are caller
 * owned: t_crow[cols+1], t_col[nnz] of A->idx_dtype, t_val[nnz] of A->val_dtype (may be NULL
 * together with A->val; must be NULL for VAL_UNIT), t_perm[nnz] int32/int64 like idx (may be
 * NULL) = source position of each transposed entry. */
OFSPMM_API size_t ofspmm_csr_transpose_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz,
                                                       int idx_dtype);
OFSPMM_API int ofspmm_csr_transpose(const ofspmm_csr* A, void* t_crow, void* t_col, void* t_val,
                                    void* t_perm, void* workspace, size_t workspace_bytes,
                                    ofspmm_stream_t stream);

/* ---- Row exchange of the multi-GPU path (SURVEY.md §8e).  `src` may be a PEER-mapped device
 * pointer (CUDA IPC / symmetric memory): the kernels read it with ordinary 16-byte loads over
 * NVLink / NVSwitch.  list == NULL means the identity (rows 0..count-1).  max_ctas caps the grid so
 * the copy shares the GPU with the product it overlaps (0: library default).
 *   gather:       dst[i, :]                       = src[list[i] - idx_offset, :]
 *   scatter-add:  dst[list[i] - idx_offset, :]   += src[i, :]      (entries of `list` distinct)
 * The reference gathers the WHOLE operand on every rank with a blocking ncclAllGather before the op
 * (oneflow/core/boxing/ccl_boxing_function.cpp:183-197, oneflow/user/kernels/nccl_logical_kernels.cpp:194-200);
 * here a rank pulls only the rows its block touches, while its local columns are already computing. */
OFSPMM_API int ofspmm_gather_rows(void* dst, int64_t ld_dst, const void* src, int64_t ld_src,
                                  const void* list, int idx_dtype, int64_t idx_offset, int64_t count,
                                  int64_t n, int dense_dtype, int max_ctas, ofspmm_stream_t stream);
OFSPMM_API int ofspmm_scatter_add_rows(void* dst, int64_t ld_dst, const void* src, int64_t ld_src,
                                       const void* list, int idx_dtype, int64_t idx_offset,
                                       int64_t count, int64_t n, int dense_dtype, int max_ctas,
                                       ofspmm_stream_t stream);

/* ---- Flag-synchronised multi-peer exchange: one launch for all peers, inter-rank ordering inside
 * the kernel.  Each rank owns a signal pad in symmetric memory; after publishing its data for
 * epoch e it writes e into its slot of every peer's pad (ofspmm_signal_peers, st.release.sys); a
 * consumer block spins on the flag of the segment it is about to read (ld.acquire.sys).  The
 * caller double-buffers the published data by epoch parity, so no "done reading" handshake exists.
 * ONE rank per GPU: kernels of different ranks wait on one another.
 *   pull:    dst[seg.dst_row + i, :] = seg.src[seg.list[i], :]          for every segment, in order
 *   combine: acc[r, :] += seg.src[seg.inv[r], :]  where seg.inv[r] >= 0, segments in the given
 *            (= rank) order: a fixed summation order; acc is fp32 (rounded once by the caller for
 *            16-bit operands, ofspmm_cast_from_f32). */
typedef struct ofspmm_pull_seg {
  const void* src;   /* peer-mapped base of the owner's published shard                         */
  const void* list;  /* device: rows wanted, relative to src (idx_dtype)                          */
  const void* flag;  /* device, uint64: THIS rank's pad slot the owner writes its epoch to        */
  int64_t count;
  int64_t dst_row;
} ofspmm_pull_seg;
typedef struct ofspmm_combine_seg {
  const void* src;   /* peer-mapped first row of the peer's partial rows for this rank's shard    */
  const void* inv;   /* device int32[rows]: this rank's row -> row of src, or -1                   */
  const void* flag;
} ofspmm_combine_seg;
OFSPMM_API int ofspmm_signal_peers(void* const* peer_slots, int n, uint64_t epoch, ofspmm_stream_t stream);
OFSPMM_API int ofspmm_pull_rows_multi(void* dst, int64_t ld_dst, int64_t ld_src, const ofspmm_pull_seg* segs,
                                      int nseg, uint64_t epoch, int64_t n, int dense_dtype, int idx_dtype,
                                      int max_ctas, ofspmm_stream_t stream);
OFSPMM_API int ofspmm_combine_rows_multi(float* acc, int64_t ld_acc, int64_t ld_src,
                                         const ofspmm_combine_seg* segs, int nseg, uint64_t epoch,
                                         int64_t rows, int64_t n, int src_dtype, int max_ctas,
                                         ofspmm_stream_t stream);

/* fp32-accumulator forms for 16-bit operands: the owner of a dB shard adds the peers' bf16 partial
 * rows into an fp32 buffer and rounds once at the end (ofspmm_cast_from_f32), instead of rounding
 * to bf16 after every rank's contribution. */
OFSPMM_API int ofspmm_scatter_add_rows_f32(float* dst, int64_t ld_dst, const void* src, int64_t ld_src,
                                           const void* list, int idx_dtype, int64_t idx_offset,
                                           int64_t count, int64_t n, int src_dtype, int max_ctas,
                                           ofspmm_stream_t stream);
OFSPMM_API int ofspmm_cast_from_f32(const float* src, void* dst, int64_t count, int dst_dtype,
                                    ofspmm_stream_t stream);

/* ---- Graph construction on the device (SURVEY.md §8f-1): the step before the path.
 * COO -> CSR: `row`, `col` int64 edge endpoints, `val` fp32 (NULL: all ones), nnz_in entries in any
 * order with duplicates.  Duplicates are merged in edge-list order — coalesce 0: sum (Graph500 /
 * scipy convention), 1: max, 2: first — and entries outside rows x cols are dropped.  Outputs:
 * crow[rows+1], col_out / val_out sized for nnz_in (only the first counts[0] entries are written),
 * columns sorted and unique within a row; counts[0] = nnz of the CSR, counts[1] = dropped entries
 * (device int64[2], may be NULL).  The caller reads counts[0] after synchronising. */
OFSPMM_API size_t ofspmm_coo_to_csr_workspace_bytes(int64_t nnz_in, int64_t rows, int64_t cols);
OFSPMM_API int ofspmm_coo_to_csr(const int64_t* row, const int64_t* col, const float* val, int64_t nnz_in,
                                 int64_t rows, int64_t cols, int coalesce, int idx_dtype, void* crow,
                                 void* col_out, float* val_out, int64_t* counts, void* workspace,
                                 size_t workspace_bytes, ofspmm_stream_t stream);
/* row_of_nnz[p] = row of stored entry p (CSR -> COO rows). */
OFSPMM_API int ofspmm_csr_expand_rows(const void* crow, int idx_dtype, int64_t rows, int64_t* row_of_nnz,
                                      ofspmm_stream_t stream);
/* In-place normalisation of fp32 values with D = diag(row sums of |A|): mode 0: D^-1/2 A D^-1/2
 * (square A, the GCN propagation matrix), mode 1: D^-1 A.  dinv_rows: `rows` floats of scratch
 * (holds the per-row scale afterwards). */
OFSPMM_API int ofspmm_csr_normalize(const void* crow, const void* col, float* val, int idx_dtype,
                                    int64_t rows, int64_t cols, int mode, float* dinv_rows,
                                    ofspmm_stream_t stream);

/* ---- Neighbour sampling (mini-batch GraphSAGE): one fan-out-sampled bipartite block of a square A
 * (rows == cols).  For destination v = dst[i] with deg = crow[v+1] - crow[v], k = deg if fanout == -1,
 * else min(deg, fanout).  Entry j of row v (0-based) has the key
 *     key(s, v, j) = mix(mix(s ^ v) + j)   (mod 2^64, compared unsigned; s = rng_seed)
 * with mix = multiply by 0x9E3779B97F4A7C15, then the splitmix64 finaliser.  The k entries with the
 * smallest (key, j) are selected: a uniform sample without replacement and a pure function of
 * (rng_seed, v, j).  A selected entry whose column lies outside [0, cols) is dropped.
 * Outputs (num_dst x num_src block, int32 blk_crow[num_dst+1] / blk_col):
 *   - row i holds the kept entries of dst[i] in ascending j; blk_val (A's value dtype; non-NULL
 *     exactly when A has values) holds val[crow[v] + j];
 *   - blk_col are LOCAL ids into src_nodes (A's index dtype, room for num_dst + cap ids):
 *     src_nodes = dst verbatim, then the distinct sampled ids that are not in dst, ascending;
 *   - counts (device int64[3]): [0] = block nnz, [1] = num_src, [2] = invalid destinations (ids
 *     outside [0, rows), and every occurrence of an id that occurs more than once; such a
 *     destination reads nothing (degree 0) and the outputs are memory-safe but meaningless).
 * `cap` is the capacity of blk_col / blk_val (cap >= 2^31-1: OFSPMM_ERR_TOO_LARGE).  If the sum of k
 * exceeds it, counts[0] reports the size needed, nothing is written past any capacity and the outputs
 * are invalid.  The workspace depends on (num_dst, cap) only, never on A's size.  num_dst == 0 writes
 * blk_crow[0] = 0 and zero counts. */
OFSPMM_API size_t ofspmm_sample_neighbors_workspace_bytes(int64_t num_dst, int64_t cap, int idx_dtype);
OFSPMM_API int ofspmm_sample_neighbors(const ofspmm_csr* A, const void* dst, int64_t num_dst, int64_t fanout,
                                       uint64_t rng_seed, int64_t cap, void* blk_crow, void* blk_col, void* blk_val,
                                       void* src_nodes, int64_t* counts, void* workspace, size_t workspace_bytes,
                                       ofspmm_stream_t stream);

/* ---- Host-buffer convenience entry (what a CPU-tensor caller / the e2e benchmark uses): copies
 * the CSR arrays and B from HOST memory (pinned recommended) to device staging carved from
 * `workspace`, runs ofspmm_fwd, copies C back to `C_host`, all on `stream`; the caller
 * synchronises the stream.  Workspace = ofspmm_fwd_host_workspace_bytes(...). */
OFSPMM_API size_t ofspmm_fwd_host_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz,
                                                  int64_t n, int dense_dtype, int idx_dtype,
                                                  int val_dtype);
OFSPMM_API int ofspmm_fwd_host(const ofspmm_csr* A_host, const void* B_host, void* C_host,
                               int64_t n, int dense_dtype, void* workspace, size_t workspace_bytes,
                               ofspmm_stream_t stream);

/* ---- Introspection. */
OFSPMM_API const char* ofspmm_strerror(int status);
OFSPMM_API int ofspmm_version(void);
/* Number of kernels the library has launched on this process so far (monotonic, relaxed atomic);
 * the benchmark reports the delta over its timed region as `gpu_launches`. */
OFSPMM_API uint64_t ofspmm_launch_count(void);
/* Name of the kernel variant ofspmm_fwd would pick for this shape (AUTO), or of an explicit
 * variant code (thread-local string, valid until the next call on the same thread). */
OFSPMM_API const char* ofspmm_fwd_variant(int64_t rows, int64_t nnz, int64_t n, int dense_dtype);
OFSPMM_API const char* ofspmm_variant_name(int variant, int64_t rows, int64_t nnz, int64_t n,
                                           int dense_dtype);

#ifdef __cplusplus
}
#endif
#endif /* OFSPMM_H_ */
