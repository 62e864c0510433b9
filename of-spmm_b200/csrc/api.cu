// api.cu — the extern "C" boundary declared in include/ofspmm.h: argument validation, workspace
// carving and dispatch to the per-op launchers.  Nothing here allocates device memory or
// synchronises; every entry point is re-entrant.
#include <stdio.h>
#include <string.h>

#include "common.cuh"
#include "internal.h"

namespace ofspmm {

std::atomic<uint64_t> g_launches{0};

int get_dev_info(DevInfo* out) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return OFSPMM_ERR_NO_DEVICE;
  // SM count / compute capability per device ordinal: immutable, memoised (sms << 8 | major)
  static std::atomic<int> memo[KernelLaunchCache::kMaxDevices];
  int packed = dev >= 0 && dev < KernelLaunchCache::kMaxDevices ? memo[dev].load(std::memory_order_relaxed) : 0;
  if (packed == 0) {
    int sms = 0, major = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return OFSPMM_ERR_CUDA;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return OFSPMM_ERR_CUDA;
    packed = (sms << 8) | (major & 0xff);
    if (dev >= 0 && dev < KernelLaunchCache::kMaxDevices) memo[dev].store(packed, std::memory_order_relaxed);
  }
  if ((packed & 0xff) != 10) return OFSPMM_ERR_NO_DEVICE;  // the library carries sm_100a code only
  out->sms = packed >> 8;
  out->cc_major = packed & 0xff;
  out->ordinal = dev;
  return OFSPMM_OK;
}

FwdWorkspace fwd_workspace_layout(int64_t rows, int64_t nnz, int64_t n, int dense_dtype, int items) {
  FwdWorkspace L;
  const size_t P = static_cast<size_t>(num_tasks(rows, nnz, items));
  const size_t rowbuf = P * static_cast<size_t>(n) * sizeof(float);
  Carve c;
  L.counter_off = c.take(256);  // task counter of the dynamic order (zeroed by a memset node before the launch)
  L.part_off = c.take((P + 1) * part_entry_bytes(nnz));
  L.carry_off = c.take(rowbuf);
  L.head_off = c.take(dense_dtype == OFSPMM_DTYPE_FLOAT ? 0 : rowbuf);
  L.total = c.total;
  return L;
}

namespace {

bool dense_ok(int d) { return d == OFSPMM_DTYPE_FLOAT || d == OFSPMM_DTYPE_BFLOAT16; }
bool idx_ok(int d) { return d == OFSPMM_DTYPE_INT32 || d == OFSPMM_DTYPE_INT64; }
size_t dense_size(int d) { return d == OFSPMM_DTYPE_FLOAT ? 4 : 2; }
size_t idx_size(int d) { return d == OFSPMM_DTYPE_INT64 ? 8 : 4; }
// Bytes per stored value: a pattern matrix (OFSPMM_VAL_UNIT) stores none.
size_t val_size(int d) { return d == OFSPMM_DTYPE_FLOAT ? 4 : (d == OFSPMM_VAL_UNIT ? 0 : 2); }
bool unit(const ofspmm_csr* A) { return A->val_dtype == OFSPMM_VAL_UNIT; }

// Sizes no kernel can address: rows that do not fit int, non-zeros that int32 row offsets cannot
// count, or more 256-item tasks than the task index allows (kMaxTasks).  Wide int64 matrices are fine.
bool too_large(int idx_dtype, int64_t rows, int64_t nnz) {
  if (rows >= (int64_t{1} << 31) - 1) return true;
  if (idx_dtype == OFSPMM_DTYPE_INT32 && wide_nnz(nnz)) return true;
  return num_tasks(rows, nnz, kTaskItems) >= kMaxTasks;
}

int check_csr(const ofspmm_csr* A, bool need_val) {
  if (A == nullptr) return OFSPMM_ERR_INVALID_ARG;
  if (A->rows < 0 || A->cols < 0 || A->nnz < 0) return OFSPMM_ERR_INVALID_ARG;
  if (!idx_ok(A->idx_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  if (A->val_dtype != OFSPMM_DTYPE_FLOAT && A->val_dtype != OFSPMM_DTYPE_BFLOAT16 && !unit(A))
    return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  if (too_large(A->idx_dtype, A->rows, A->nnz)) return OFSPMM_ERR_TOO_LARGE;
  if (A->crow == nullptr) return OFSPMM_ERR_INVALID_ARG;
  if (unit(A) && A->val != nullptr) return OFSPMM_ERR_INVALID_ARG;  // a values array with the pattern dtype
  if (A->nnz > 0 && (A->col == nullptr || (need_val && !unit(A) && A->val == nullptr))) return OFSPMM_ERR_INVALID_ARG;
  return OFSPMM_OK;
}

int check_dtypes(const ofspmm_csr* A, int dense_dtype) {
  if (!dense_ok(dense_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  if (A->val_dtype == OFSPMM_DTYPE_BFLOAT16 && dense_dtype != OFSPMM_DTYPE_BFLOAT16) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  return OFSPMM_OK;
}

// Checks of a product's A, dense dtype and width n.
int check_product(const ofspmm_csr* A, bool need_val, int dense_dtype, int64_t n) {
  if (int rc = check_csr(A, need_val)) return rc;
  if (int rc = check_dtypes(A, dense_dtype)) return rc;
  if (n < 0 || n >= (int64_t{1} << 31)) return OFSPMM_ERR_INVALID_ARG;
  return OFSPMM_OK;
}

// Checks of the forward entry points: B may be NULL when no non-zero reads it.
int check_fwd(const ofspmm_csr* A, const void* B, const void* C, int64_t n, int dense_dtype) {
  if (int rc = check_product(A, true, dense_dtype, n)) return rc;
  if (A->rows > 0 && n > 0 && (C == nullptr || (A->nnz > 0 && A->cols > 0 && B == nullptr))) return OFSPMM_ERR_INVALID_ARG;
  return OFSPMM_OK;
}

// Checks of the A^T·dY entry points and the calls that need no product; *done: dB is complete,
// because it has no elements or because A is empty and `zero_empty` zeroed it.
int begin_bwd(const ofspmm_csr* A, const void* dY, void* dB, int64_t n, int dense_dtype, bool zero_empty,
              cudaStream_t stream, bool* done) {
  *done = true;
  if (int rc = check_product(A, true, dense_dtype, n)) return rc;
  if (A->cols == 0 || n == 0) return OFSPMM_OK;
  if (dB == nullptr || (A->nnz > 0 && dY == nullptr)) return OFSPMM_ERR_INVALID_ARG;
  if (zero_empty && (A->nnz == 0 || A->rows == 0)) {
    OFSPMM_CUDA_OK(cudaMemsetAsync(dB, 0, static_cast<size_t>(A->cols) * n * dense_size(dense_dtype), stream));
    return OFSPMM_OK;
  }
  *done = false;
  return OFSPMM_OK;
}

// Checks of the sampling options (NULL: none): known flags only; weights of a dense dtype, and not
// with replacement; an exclusion list of a non-negative size, present unless empty.
int check_sample_opts(const ofspmm_sample_opts* o) {
  if (o == nullptr) return OFSPMM_OK;
  if (o->flags & ~static_cast<uint32_t>(OFSPMM_SAMPLE_REPLACE | OFSPMM_SAMPLE_EDGE_IDS | OFSPMM_SAMPLE_EXCLUDE))
    return OFSPMM_ERR_INVALID_ARG;
  if (o->prob != nullptr && ((o->flags & OFSPMM_SAMPLE_REPLACE) || !dense_ok(o->prob_dtype))) return OFSPMM_ERR_INVALID_ARG;
  if ((o->flags & OFSPMM_SAMPLE_EXCLUDE) && (o->num_exclude < 0 || (o->num_exclude > 0 && o->exclude == nullptr)))
    return OFSPMM_ERR_INVALID_ARG;
  return OFSPMM_OK;
}
bool sample_edge_ids(const ofspmm_sample_opts* o) { return o != nullptr && (o->flags & OFSPMM_SAMPLE_EDGE_IDS); }

int check_ws(const void* ws, size_t have, size_t need) {
  if (need == 0) return OFSPMM_OK;
  if (ws == nullptr || have < need) return OFSPMM_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(ws) & 15) return OFSPMM_ERR_WORKSPACE;
  return OFSPMM_OK;
}

// Forward workspace of a call that leaves the variant to the library (AUTO).
size_t fwd_ws_auto(int64_t rows, int64_t nnz, int64_t n, int dense_dtype) {
  return fwd_workspace_layout(rows, nnz, n, dense_dtype,
                              resolve_variant(OFSPMM_VARIANT_AUTO, rows, nnz, n, dense_dtype).items).total;
}

size_t plan_bytes_for(int64_t rows, int64_t nnz, int items) {
  return align_up((static_cast<size_t>(num_tasks(rows, nnz, items)) + 1) * part_entry_bytes(nnz), 256);
}

// Layout of the atomic route of ofspmm_bwd_b: [task partition | fp32 accumulator of a 16-bit dB]
struct AtomicLayout {
  size_t part, acc, total;
};
AtomicLayout atomic_layout(int64_t rows, int64_t cols, int64_t nnz, int64_t n, int dense_dtype) {
  AtomicLayout L;
  Carve c;
  L.part = c.take(plan_bytes_for(rows, nnz, kTaskItems));
  L.acc = c.take(dense_dtype == OFSPMM_DTYPE_FLOAT ? 0 : static_cast<size_t>(cols) * n * sizeof(float));
  L.total = c.total;
  return L;
}

// Layout of the transient-transpose route: [t_crow | t_col | t_val | transpose scratch | fwd scratch]
struct TransientLayout {
  size_t t_crow, t_col, t_val, tws, tws_bytes, fws, total;
};
TransientLayout transient_layout(int64_t rows, int64_t cols, int64_t nnz, int64_t n, int dense_dtype,
                                 int idx_dtype, int val_dtype) {
  TransientLayout L;
  const size_t is = idx_size(idx_dtype), entries = static_cast<size_t>(nnz > 0 ? nnz : 1);
  Carve c;
  L.t_crow = c.take(static_cast<size_t>(cols + 1) * is);
  L.t_col = c.take(entries * is);
  L.t_val = c.take(entries * val_size(val_dtype));  // 0 for a pattern matrix
  L.tws_bytes = transpose_workspace_bytes(rows, cols, nnz, idx_dtype);
  L.tws = c.take(L.tws_bytes);
  L.fws = c.take(fwd_ws_auto(cols, nnz, n, dense_dtype));
  L.total = c.total;
  return L;
}

// Layout of the cached-transpose route: [values of A^T | fwd scratch]
struct CachedLayout {
  size_t t_val, fws, total;
};
CachedLayout cached_layout(int64_t cols, int64_t nnz, int64_t n, int dense_dtype, int val_dtype) {
  CachedLayout L;
  Carve c;
  L.t_val = c.take(static_cast<size_t>(nnz > 0 ? nnz : 1) * val_size(val_dtype));
  L.fws = c.take(fwd_ws_auto(cols, nnz, n, dense_dtype));
  L.total = c.total;
  return L;
}

// Layout of the SDDMM: [task counter | task partition]
struct SddmmLayout {
  size_t counter, part, total;
};
SddmmLayout sddmm_layout(int64_t rows, int64_t nnz) {
  SddmmLayout L;
  Carve c;
  L.counter = c.take(256);
  L.part = c.take(plan_bytes_for(rows, nnz, kTaskItems));
  L.total = c.total;
  return L;
}

// Layout of ofspmm_fwd_host: [crow | col | val | B | C | fwd scratch], the operands staged on the device
struct HostFwdLayout {
  size_t crow, col, val, B, C, fws, total;
};
HostFwdLayout host_fwd_layout(int64_t rows, int64_t cols, int64_t nnz, int64_t n, int dense_dtype, int idx_dtype,
                              int val_dtype) {
  HostFwdLayout L;
  const size_t is = idx_size(idx_dtype), ds = dense_size(dense_dtype);
  Carve c;
  L.crow = c.take(static_cast<size_t>(rows + 1) * is);
  L.col = c.take(static_cast<size_t>(nnz) * is);
  L.val = c.take(static_cast<size_t>(nnz) * val_size(val_dtype));
  L.B = c.take(static_cast<size_t>(cols) * n * ds);
  L.C = c.take(static_cast<size_t>(rows) * n * ds);
  L.fws = c.take(fwd_ws_auto(rows, nnz, n, dense_dtype));
  L.total = c.total;
  return L;
}

// Options of one call -> launch description.  `opts` may be NULL (all defaults).
FwdLaunch make_launch(const ofspmm_opts* opts, int64_t rows, int64_t nnz, int64_t n, int dense_dtype) {
  FwdLaunch L;
  L.variant = resolve_variant(opts ? opts->variant : OFSPMM_VARIANT_AUTO, rows, nnz, n, dense_dtype);
  L.tasks_per_warp = opts && opts->tasks_per_warp > 0 ? opts->tasks_per_warp : 0;
  L.reserve_ctas = opts && opts->reserve_ctas_per_sm > 0 ? opts->reserve_ctas_per_sm : 0;
  const uint32_t fl = opts ? opts->flags : 0u;
  // task order: dynamic (drawn from a counter) unless the caller pins the static interleave
  L.dynamic = OFSPMM_DEFAULT_DYNAMIC_ORDER ? (fl & OFSPMM_ORDER_STATIC) == 0 : (fl & OFSPMM_ORDER_DYNAMIC) != 0;
  L.wide = wide_nnz(nnz);
  L.flags = fl & (OFSPMM_FWD_ACCUMULATE | OFSPMM_FWD_BIAS | OFSPMM_FWD_RELU | OFSPMM_FWD_ACC32_IN | OFSPMM_FWD_ACC32_OUT |
                 OFSPMM_FWD_MEAN);
  L.bias = opts ? opts->bias : nullptr;
  L.acc32 = opts ? static_cast<float*>(opts->acc32) : nullptr;
  return L;
}

// C = A·B through the merge-path kernels; shared by every forward-shaped entry point.
int run_fwd(const ofspmm_csr* A, const void* B, int64_t ldb, void* C, int64_t ldc, int64_t n,
            int dense_dtype, const ofspmm_opts* opts, void* ws, size_t ws_bytes, cudaStream_t stream) {
  // the mean divides this call's complete row sum: with an accumulated C (or fp32 row sums carried
  // between passes) the division would also apply to what earlier passes added
  if (opts != nullptr && (opts->flags & OFSPMM_FWD_MEAN) &&
      (opts->flags & (OFSPMM_FWD_ACCUMULATE | OFSPMM_FWD_ACC32_IN | OFSPMM_FWD_ACC32_OUT)))
    return OFSPMM_ERR_INVALID_ARG;
  if (A->rows == 0 || n == 0) return OFSPMM_OK;
  if (ldb < n || ldc < n || ldb >= (int64_t{1} << 30)) return OFSPMM_ERR_INVALID_ARG;
  FwdLaunch L = make_launch(opts, A->rows, A->nnz, n, dense_dtype);
  if ((L.flags & OFSPMM_FWD_BIAS) && L.bias == nullptr) return OFSPMM_ERR_INVALID_ARG;
  if (L.flags & (OFSPMM_FWD_ACC32_IN | OFSPMM_FWD_ACC32_OUT)) {
    // fp32 row accumulator between the passes of a 16-bit product (fp32 products accumulate in C)
    if (dense_dtype == OFSPMM_DTYPE_FLOAT || L.acc32 == nullptr || (reinterpret_cast<uintptr_t>(L.acc32) & 15) ||
        (L.flags & OFSPMM_FWD_ACCUMULATE))
      return OFSPMM_ERR_INVALID_ARG;
  }
  if (A->nnz == 0 || A->cols == 0) {
    // every row sum is 0, and so is its mean: MEAN changes nothing here
    const unsigned fl = L.flags & ~static_cast<unsigned>(OFSPMM_FWD_MEAN);
    if (fl == OFSPMM_FWD_ACCUMULATE || fl == (OFSPMM_FWD_ACC32_IN | OFSPMM_FWD_ACC32_OUT)) return OFSPMM_OK;  // += 0
    if (fl == 0) {
      OFSPMM_CUDA_OK(cudaMemset2DAsync(C, static_cast<size_t>(ldc) * dense_size(dense_dtype), 0,
                                       static_cast<size_t>(n) * dense_size(dense_dtype),
                                       static_cast<size_t>(A->rows), stream));
      return OFSPMM_OK;
    }
    // bias / relu of an all-zero product: run the kernels on the (empty) rows; needs a valid crow
    if (A->nnz != 0) return OFSPMM_ERR_INVALID_ARG;
  }
  const FwdWorkspace W = fwd_workspace_layout(A->rows, A->nnz, n, dense_dtype, L.variant.items);
  if (int rc = check_ws(ws, ws_bytes, W.total)) return rc;
  unsigned char* w = static_cast<unsigned char*>(ws);
  const int64_t P = num_tasks(A->rows, A->nnz, L.variant.items);
  const void* part = w + W.part_off;
  if (opts != nullptr && opts->plan != nullptr) {
    // a plan built for another task size is a caller bug, not something to paper over
    if (opts->plan_bytes != plan_bytes_for(A->rows, A->nnz, L.variant.items)) return OFSPMM_ERR_INVALID_ARG;
    part = opts->plan;
  } else if (rows_kernel_applies(A, B, ldb, C, ldc, n, dense_dtype, L)) {
    part = nullptr;  // the whole-row kernel reads crow directly: no task list
  } else if (int rc = launch_task_partition(A->crow, A->idx_dtype, A->rows, A->nnz, P, L.variant.items,
                                            w + W.part_off, stream)) {
    return rc;
  }
  return launch_fwd(A, B, ldb, C, ldc, n, dense_dtype, part, reinterpret_cast<float*>(w + W.carry_off),
                    reinterpret_cast<float*>(w + W.head_off), w + W.counter_off, P, L, stream);
}

}  // namespace
}  // namespace ofspmm

using namespace ofspmm;

extern "C" {

size_t ofspmm_fwd_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int64_t n, int dense_dtype) {
  return ofspmm_fwd_ex_workspace_bytes(rows, cols, nnz, n, dense_dtype, OFSPMM_VARIANT_AUTO);
}

size_t ofspmm_fwd_ex_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int64_t n, int dense_dtype,
                                     int variant) {
  (void)cols;
  if (rows < 0 || nnz < 0 || n < 0) return 0;
  return fwd_workspace_layout(rows, nnz, n, dense_dtype, resolve_variant(variant, rows, nnz, n, dense_dtype).items).total;
}

int ofspmm_fwd_ex(const ofspmm_csr* A, const void* B, int64_t ldb, void* C, int64_t ldc, int64_t n,
                  int dense_dtype, const ofspmm_opts* opts, void* workspace, size_t workspace_bytes,
                  ofspmm_stream_t stream) {
  if (int rc = check_fwd(A, B, C, n, dense_dtype)) return rc;
  return run_fwd(A, B, ldb, C, ldc, n, dense_dtype, opts, workspace, workspace_bytes, reinterpret_cast<cudaStream_t>(stream));
}

size_t ofspmm_plan_bytes(int64_t rows, int64_t nnz, int64_t n, int dense_dtype, int variant) {
  if (rows < 0 || nnz < 0) return 0;
  return plan_bytes_for(rows, nnz, resolve_variant(variant, rows, nnz, n, dense_dtype).items);
}

int ofspmm_plan_build(const void* crow, int idx_dtype, int64_t rows, int64_t nnz, int64_t n, int dense_dtype,
                      int variant, void* plan, size_t plan_bytes, ofspmm_stream_t stream) {
  if (crow == nullptr || plan == nullptr || rows < 0 || nnz < 0) return OFSPMM_ERR_INVALID_ARG;
  if (!idx_ok(idx_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  if (too_large(idx_dtype, rows, nnz)) return OFSPMM_ERR_TOO_LARGE;
  const int items = resolve_variant(variant, rows, nnz, n, dense_dtype).items;
  if (plan_bytes < plan_bytes_for(rows, nnz, items) || (reinterpret_cast<uintptr_t>(plan) & 15)) return OFSPMM_ERR_WORKSPACE;
  return launch_task_partition(crow, idx_dtype, rows, nnz, num_tasks(rows, nnz, items), items, plan,
                               reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_choose_variant(const int64_t* hist32_host, int64_t rows, int64_t nnz, int64_t n, int dense_dtype) {
  FwdVariant v = resolve_variant(OFSPMM_VARIANT_AUTO, rows, nnz, n, dense_dtype);
  if (hist32_host == nullptr || rows <= 0 || nnz <= 0) return encode_variant(v);
  if (v.items == kSmallTaskItems) {
    // Small problem (fewer 256-item tasks than resident warps): launch, staging and carry
    // latencies dominate.  If no row reaches 512 non-zeros (histogram buckets >= 10 empty) and one
    // lane group per row yields at least 8 warps per SM, the whole-row kernel does the product in
    // ONE launch (cfg1: 34.6 -> see profiles/r2_cfg1_latency.md); otherwise 64-item tasks.
    int64_t long_rows = 0;
    for (int b = 10; b < 32; ++b) long_rows += hist32_host[b];
    const LaneLayout rl = lane_layout(LaneOp::kFwdRows, dense_dtype, n, true);
    if (rl.ok() && long_rows == 0) {
      const int64_t warps = (rows * rl.lpr + 31) / 32;
      if (warps >= 148 * 8) return encode_variant(resolve_variant(OFSPMM_VARIANT_EXPLICIT | OFSPMM_VARIANT_ROWS, rows, nnz, n, dense_dtype));
    }
    return encode_variant(v);
  }
  // Row-parallel groups (each 8 / 16-lane group owns whole rows, 4 / 2 rows in flight per warp)
  // against nnz-parallel groups (every group works on every row): measured on B200 at N = 32 / 64
  // fp32, the row-parallel layout wins 10-20 % on R-MAT (median row length 0-1, 90 % of the rows
  // under 16 non-zeros) and loses 5 % on products-shaped (median 32-63) and 60 % on Reddit-shaped
  // rows (median 256-511), where one long row piece leaves three of four groups idle
  // (profiles/r2_variant_sweeps.md).  Criterion: the MEDIAN row, empty rows included, has fewer
  // than 16 non-zeros, i.e. the per-row work dominates the per-non-zero work.
  const bool sub_warp_rows = lane_layout(LaneOp::kFwdRowPar, dense_dtype, n, true).ok();
  int64_t below16 = 0;
  for (int b = 0; b <= 4; ++b) below16 += hist32_host[b];  // buckets 0..4 = lengths 0..15
  v.row_parallel = sub_warp_rows && 2 * below16 > rows;
  // resolve again so unsupported widths fall back exactly as the launch would
  return encode_variant(resolve_variant(encode_variant(v), rows, nnz, n, dense_dtype));
}

int ofspmm_fwd(const ofspmm_csr* A, const void* B, void* C, int64_t n, int dense_dtype, void* workspace,
               size_t workspace_bytes, ofspmm_stream_t stream) {
  return ofspmm_fwd_ex(A, B, n, C, n, n, dense_dtype, nullptr, workspace, workspace_bytes, stream);
}

int ofspmm_fwd_strided(const ofspmm_csr* A, const void* B, int64_t ldb, void* C, int64_t ldc, int64_t n,
                       int dense_dtype, void* workspace, size_t workspace_bytes, ofspmm_stream_t stream) {
  return ofspmm_fwd_ex(A, B, ldb, C, ldc, n, dense_dtype, nullptr, workspace, workspace_bytes, stream);
}

size_t ofspmm_bwd_b_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int64_t n, int dense_dtype,
                                    int have_transpose) {
  if (rows < 0 || cols < 0 || nnz < 0 || n < 0) return 0;
  if (have_transpose) return fwd_ws_auto(cols, nnz, n, dense_dtype);
  return atomic_layout(rows, cols, nnz, n, dense_dtype).total;
}

int ofspmm_bwd_b(const ofspmm_csr* A, const ofspmm_csr* At, const void* dY, void* dB, int64_t n,
                 int dense_dtype, void* workspace, size_t workspace_bytes, ofspmm_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  bool done;
  // route (1) runs the forward kernel on A^T even when A is empty
  if (int rc = begin_bwd(A, dY, dB, n, dense_dtype, At == nullptr, stream, &done); rc != OFSPMM_OK || done) return rc;
  if (At != nullptr) {  // route (1): forward kernel on the cached transpose
    if (int rc = check_csr(At, true)) return rc;
    if (At->rows != A->cols || At->cols != A->rows || At->nnz != A->nnz) return OFSPMM_ERR_INVALID_ARG;
    if (int rc = check_dtypes(At, dense_dtype)) return rc;
    return run_fwd(At, dY, n, dB, n, n, dense_dtype, nullptr, workspace, workspace_bytes, stream);
  }
  // route (2): vector-atomic scatter into an fp32 accumulator
  const AtomicLayout L = atomic_layout(A->rows, A->cols, A->nnz, n, dense_dtype);
  if (int rc = check_ws(workspace, workspace_bytes, L.total)) return rc;
  unsigned char* w = static_cast<unsigned char*>(workspace);
  const int64_t P = num_tasks(A->rows, A->nnz);
  if (int rc = launch_task_partition(A->crow, A->idx_dtype, A->rows, A->nnz, P, kTaskItems, w + L.part, stream)) return rc;
  if (dense_dtype == OFSPMM_DTYPE_FLOAT)
    return launch_bwd_atomic(A, dY, static_cast<float*>(dB), nullptr, n, dense_dtype, w + L.part, P, stream);
  return launch_bwd_atomic(A, dY, reinterpret_cast<float*>(w + L.acc), dB, n, dense_dtype, w + L.part, P, stream);
}

size_t ofspmm_bwd_b_transient_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int64_t n,
                                              int dense_dtype, int idx_dtype, int val_dtype) {
  if (rows < 0 || cols < 0 || nnz < 0 || n < 0 || !idx_ok(idx_dtype)) return 0;
  return transient_layout(rows, cols, nnz, n, dense_dtype, idx_dtype, val_dtype).total;
}

int ofspmm_bwd_b_transient(const ofspmm_csr* A, const void* dY, void* dB, int64_t n, int dense_dtype,
                           void* workspace, size_t workspace_bytes, ofspmm_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  bool done;
  if (int rc = begin_bwd(A, dY, dB, n, dense_dtype, true, stream, &done); rc != OFSPMM_OK || done) return rc;
  const TransientLayout L = transient_layout(A->rows, A->cols, A->nnz, n, dense_dtype, A->idx_dtype, A->val_dtype);
  if (int rc = check_ws(workspace, workspace_bytes, L.total)) return rc;
  unsigned char* w = static_cast<unsigned char*>(workspace);
  void* t_val = unit(A) ? nullptr : w + L.t_val;  // a pattern A^T has no values to build
  if (int rc = launch_transpose(A, w + L.t_crow, w + L.t_col, t_val, nullptr, w + L.tws, L.tws_bytes, stream)) return rc;
  ofspmm_csr At = *A;
  At.rows = A->cols;
  At.cols = A->rows;
  At.crow = w + L.t_crow;
  At.col = w + L.t_col;
  At.val = t_val;
  return run_fwd(&At, dY, n, dB, n, n, dense_dtype, nullptr, w + L.fws, workspace_bytes - L.fws, stream);
}

size_t ofspmm_bwd_b_cached_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int64_t n, int dense_dtype,
                                          int val_dtype) {
  if (rows < 0 || cols < 0 || nnz < 0 || n < 0) return 0;
  return cached_layout(cols, nnz, n, dense_dtype, val_dtype).total;
}

int ofspmm_bwd_b_cached(const ofspmm_csr* A, const void* t_crow, const void* t_col, const void* t_perm,
                        const void* dY, void* dB, int64_t n, int dense_dtype, const ofspmm_opts* opts,
                        void* workspace, size_t workspace_bytes, ofspmm_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  bool done;
  // an empty A runs the forward kernel, which writes the zeros of dB
  if (int rc = begin_bwd(A, dY, dB, n, dense_dtype, false, stream, &done); rc != OFSPMM_OK || done) return rc;
  if (t_crow == nullptr || (A->nnz > 0 && (t_col == nullptr || t_perm == nullptr))) return OFSPMM_ERR_INVALID_ARG;
  const CachedLayout L = cached_layout(A->cols, A->nnz, n, dense_dtype, A->val_dtype);
  if (int rc = check_ws(workspace, workspace_bytes, L.total)) return rc;
  unsigned char* w = static_cast<unsigned char*>(workspace);
  // the STRUCTURE of A^T is cached by the caller; the values are re-gathered from A on every call,
  // so in-place updates of a_val (learnable edge weights) are always seen.  A pattern matrix has
  // nothing to gather.
  if (!unit(A))
    if (int rc = launch_gather_vals(A->val, A->val_dtype, t_perm, A->idx_dtype, A->nnz, w + L.t_val, stream)) return rc;
  ofspmm_csr At = *A;
  At.rows = A->cols;
  At.cols = A->rows;
  At.crow = t_crow;
  At.col = t_col;
  At.val = unit(A) ? nullptr : w + L.t_val;
  return run_fwd(&At, dY, n, dB, n, n, dense_dtype, opts, w + L.fws, workspace_bytes - L.fws, stream);
}

size_t ofspmm_coo_to_csr_workspace_bytes(int64_t nnz_in, int64_t rows, int64_t cols) {
  if (nnz_in < 0 || rows < 0 || cols < 0) return 0;
  return coo_to_csr_workspace_bytes(nnz_in, rows, cols);
}

int ofspmm_coo_to_csr(const int64_t* row, const int64_t* col, const float* val, int64_t nnz_in, int64_t rows, int64_t cols,
                      int coalesce, int idx_dtype, void* crow, void* col_out, float* val_out, int64_t* counts,
                      void* workspace, size_t workspace_bytes, ofspmm_stream_t stream) {
  if (nnz_in < 0 || rows < 0 || cols < 0 || coalesce < 0 || coalesce > 2) return OFSPMM_ERR_INVALID_ARG;
  if (crow == nullptr || (nnz_in > 0 && (row == nullptr || col == nullptr || col_out == nullptr || val_out == nullptr)))
    return OFSPMM_ERR_INVALID_ARG;
  if (!idx_ok(idx_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  if (nnz_in >= (int64_t{1} << 31) - 1) return OFSPMM_ERR_TOO_LARGE;
  if (rows > 0 && cols > 0 && rows > ((int64_t{1} << 62) / cols)) return OFSPMM_ERR_TOO_LARGE;   // row*cols+col must fit
  return launch_coo_to_csr(row, col, val, nnz_in, rows, cols, coalesce, idx_dtype, crow, col_out, val_out, counts, workspace,
                           workspace_bytes, reinterpret_cast<cudaStream_t>(stream));
}

size_t ofspmm_sample_neighbors_workspace_bytes(int64_t num_dst, int64_t cap, int idx_dtype) {
  return ofspmm_sample_neighbors_ex_workspace_bytes(num_dst, cap, idx_dtype, nullptr);
}

size_t ofspmm_sample_neighbors_ex_workspace_bytes(int64_t num_dst, int64_t cap, int idx_dtype,
                                                  const ofspmm_sample_opts* opts) {
  if (num_dst < 0 || cap < 0 || !idx_ok(idx_dtype) || check_sample_opts(opts) != OFSPMM_OK) return 0;
  return sample_neighbors_workspace_bytes(num_dst, cap, sample_edge_ids(opts));
}

int ofspmm_sample_neighbors(const ofspmm_csr* A, const void* dst, int64_t num_dst, int64_t fanout, uint64_t rng_seed,
                            int64_t cap, void* blk_crow, void* blk_col, void* blk_val, void* src_nodes, int64_t* counts,
                            void* workspace, size_t workspace_bytes, ofspmm_stream_t stream) {
  return ofspmm_sample_neighbors_ex(A, nullptr, dst, num_dst, fanout, rng_seed, cap, blk_crow, blk_col, blk_val, nullptr,
                                    src_nodes, counts, workspace, workspace_bytes, stream);
}

int ofspmm_sample_neighbors_ex(const ofspmm_csr* A, const ofspmm_sample_opts* opts, const void* dst, int64_t num_dst,
                               int64_t fanout, uint64_t rng_seed, int64_t cap, void* blk_crow, void* blk_col,
                               void* blk_val, void* blk_eid, void* src_nodes, int64_t* counts, void* workspace,
                               size_t workspace_bytes, ofspmm_stream_t stream) {
  if (int rc = check_csr(A, true)) return rc;
  if (A->rows != A->cols || fanout < -1 || num_dst < 0 || cap < 0) return OFSPMM_ERR_INVALID_ARG;
  if (cap >= kWideNnz || num_dst >= kWideNnz) return OFSPMM_ERR_TOO_LARGE;   // int32 block offsets and local ids
  if (blk_crow == nullptr || counts == nullptr) return OFSPMM_ERR_INVALID_ARG;
  if (num_dst > 0 && (dst == nullptr || src_nodes == nullptr)) return OFSPMM_ERR_INVALID_ARG;
  if (cap > 0 && (blk_col == nullptr || src_nodes == nullptr)) return OFSPMM_ERR_INVALID_ARG;
  // a values array exactly when A has values (a forgotten value dtype is caught, not ignored)
  if (unit(A) ? blk_val != nullptr : (cap > 0 && blk_val == nullptr)) return OFSPMM_ERR_INVALID_ARG;
  if (int rc = check_sample_opts(opts)) return rc;
  // an edge-id array exactly when asked for
  const bool eid = sample_edge_ids(opts);
  if (eid ? (cap > 0 && blk_eid == nullptr) : blk_eid != nullptr) return OFSPMM_ERR_INVALID_ARG;
  if (int rc = check_ws(workspace, workspace_bytes, sample_neighbors_workspace_bytes(num_dst, cap, eid))) return rc;
  return launch_sample_neighbors(A, opts, dst, num_dst, fanout, rng_seed, cap, blk_crow, blk_col, blk_val,
                                 eid ? blk_eid : nullptr, src_nodes, counts, workspace,
                                 reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_edge_ids(const ofspmm_csr* A, const void* u, const void* v, int64_t n, void* eid, ofspmm_stream_t stream) {
  if (int rc = check_csr(A, false)) return rc;
  if (n < 0 || (n > 0 && (u == nullptr || v == nullptr || eid == nullptr))) return OFSPMM_ERR_INVALID_ARG;
  return launch_edge_ids(A, u, v, n, eid, reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_negative_sample(const ofspmm_csr* A, const void* src, int64_t num_src, int64_t k, uint64_t rng_seed,
                           uint32_t flags, int32_t max_trials, void* neg_dst, int64_t* counts, ofspmm_stream_t stream) {
  if (int rc = check_csr(A, false)) return rc;
  if (num_src < 0 || k < 0 || max_trials < 1 || counts == nullptr) return OFSPMM_ERR_INVALID_ARG;
  if (flags & ~static_cast<uint32_t>(OFSPMM_NEG_EXCLUDE_EDGES | OFSPMM_NEG_EXCLUDE_SELF)) return OFSPMM_ERR_INVALID_ARG;
  if ((flags & OFSPMM_NEG_EXCLUDE_SELF) && A->rows != A->cols) return OFSPMM_ERR_INVALID_ARG;
  if (k > 0 && num_src > INT64_MAX / k) return OFSPMM_ERR_TOO_LARGE;   // num_src * k slots must be addressable
  if (num_src > 0 && (src == nullptr || (k > 0 && neg_dst == nullptr))) return OFSPMM_ERR_INVALID_ARG;
  return launch_negative_sample(A, src, num_src, k, rng_seed, flags, max_trials, neg_dst, counts,
                                reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_csr_expand_rows(const void* crow, int idx_dtype, int64_t rows, int64_t* row_of_nnz, ofspmm_stream_t stream) {
  if (rows < 0 || crow == nullptr || (rows > 0 && row_of_nnz == nullptr)) return OFSPMM_ERR_INVALID_ARG;
  if (!idx_ok(idx_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  return launch_expand_rows(crow, idx_dtype, rows, row_of_nnz, reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_csr_normalize(const void* crow, const void* col, float* val, int idx_dtype, int64_t rows, int64_t cols, int mode,
                         float* dinv_rows, ofspmm_stream_t stream) {
  if (rows < 0 || cols < 0 || crow == nullptr || (mode != 0 && mode != 1)) return OFSPMM_ERR_INVALID_ARG;
  if (rows > 0 && dinv_rows == nullptr) return OFSPMM_ERR_WORKSPACE;
  if (mode == 0 && rows != cols) return OFSPMM_ERR_INVALID_ARG;   // D^-1/2 A D^-1/2 needs a square matrix
  if (!idx_ok(idx_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  return launch_csr_normalize(crow, col, val, idx_dtype, rows, cols, mode, dinv_rows, reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_permute_values(const void* val, int val_dtype, const void* perm, int idx_dtype, int64_t nnz, void* out,
                          ofspmm_stream_t stream) {
  if (nnz < 0) return OFSPMM_ERR_INVALID_ARG;
  if (nnz > 0 && (val == nullptr || perm == nullptr || out == nullptr)) return OFSPMM_ERR_INVALID_ARG;
  if (!idx_ok(idx_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  return launch_gather_vals(val, val_dtype, perm, idx_dtype, nnz, out, reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_gather_rows(void* dst, int64_t ld_dst, const void* src, int64_t ld_src, const void* list, int idx_dtype,
                       int64_t idx_offset, int64_t count, int64_t n, int dense_dtype, int max_ctas,
                       ofspmm_stream_t stream) {
  if (count < 0 || n < 0 || ld_dst < n || ld_src < n) return OFSPMM_ERR_INVALID_ARG;
  if (count > 0 && n > 0 && (dst == nullptr || src == nullptr)) return OFSPMM_ERR_INVALID_ARG;
  if (list != nullptr && !idx_ok(idx_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  return launch_gather_rows(dst, ld_dst, src, ld_src, list, list ? idx_dtype : OFSPMM_DTYPE_INT32, idx_offset, count, n,
                            dense_dtype, max_ctas, reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_signal_peers(void* const* peer_slots, int n, uint64_t epoch, ofspmm_stream_t stream) {
  if (n < 0 || (n > 0 && peer_slots == nullptr)) return OFSPMM_ERR_INVALID_ARG;
  for (int i = 0; i < n; ++i)
    if (peer_slots[i] == nullptr) return OFSPMM_ERR_INVALID_ARG;
  return launch_signal_peers(peer_slots, n, epoch, reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_pull_rows_multi(void* dst, int64_t ld_dst, int64_t ld_src, const ofspmm_pull_seg* segs, int nseg,
                           uint64_t epoch, int64_t n, int dense_dtype, int idx_dtype, int max_ctas,
                           ofspmm_stream_t stream) {
  if (n < 0 || ld_dst < n || ld_src < n || nseg < 0 || (nseg > 0 && (segs == nullptr || dst == nullptr)))
    return OFSPMM_ERR_INVALID_ARG;
  return launch_pull_rows_multi(dst, ld_dst, ld_src, segs, nseg, epoch, n, dense_dtype, idx_dtype, max_ctas,
                                reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_combine_rows_multi(float* acc, int64_t ld_acc, int64_t ld_src, const ofspmm_combine_seg* segs, int nseg,
                              uint64_t epoch, int64_t rows, int64_t n, int src_dtype, int max_ctas,
                              ofspmm_stream_t stream) {
  if (n < 0 || rows < 0 || ld_acc < n || ld_src < n || nseg < 0 || (nseg > 0 && (segs == nullptr || acc == nullptr)))
    return OFSPMM_ERR_INVALID_ARG;
  return launch_combine_rows_multi(acc, ld_acc, ld_src, segs, nseg, epoch, rows, n, src_dtype, max_ctas,
                                   reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_scatter_add_rows_f32(float* dst, int64_t ld_dst, const void* src, int64_t ld_src, const void* list,
                                int idx_dtype, int64_t idx_offset, int64_t count, int64_t n, int src_dtype,
                                int max_ctas, ofspmm_stream_t stream) {
  if (count < 0 || n < 0 || ld_dst < n || ld_src < n) return OFSPMM_ERR_INVALID_ARG;
  if (count > 0 && n > 0 && (dst == nullptr || src == nullptr)) return OFSPMM_ERR_INVALID_ARG;
  if (list != nullptr && !idx_ok(idx_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  return launch_scatter_add_rows_f32(dst, ld_dst, src, ld_src, list, list ? idx_dtype : OFSPMM_DTYPE_INT32, idx_offset,
                                     count, n, src_dtype, max_ctas, reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_cast_from_f32(const float* src, void* dst, int64_t count, int dst_dtype, ofspmm_stream_t stream) {
  if (count < 0 || (count > 0 && (src == nullptr || dst == nullptr))) return OFSPMM_ERR_INVALID_ARG;
  return launch_cast_from_f32(src, dst, count, dst_dtype, reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_scatter_add_rows(void* dst, int64_t ld_dst, const void* src, int64_t ld_src, const void* list,
                            int idx_dtype, int64_t idx_offset, int64_t count, int64_t n, int dense_dtype,
                            int max_ctas, ofspmm_stream_t stream) {
  if (count < 0 || n < 0 || ld_dst < n || ld_src < n) return OFSPMM_ERR_INVALID_ARG;
  if (count > 0 && n > 0 && (dst == nullptr || src == nullptr)) return OFSPMM_ERR_INVALID_ARG;
  if (list != nullptr && !idx_ok(idx_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  return launch_scatter_add_rows(dst, ld_dst, src, ld_src, list, list ? idx_dtype : OFSPMM_DTYPE_INT32, idx_offset, count,
                                 n, dense_dtype, max_ctas, reinterpret_cast<cudaStream_t>(stream));
}

size_t ofspmm_sddmm_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int64_t n, int dense_dtype) {
  (void)cols; (void)n; (void)dense_dtype;
  if (rows < 0 || nnz < 0) return 0;
  return sddmm_layout(rows, nnz).total;
}

int ofspmm_sddmm(const ofspmm_csr* A, const void* dY, const void* B, void* dval, int64_t n, int dense_dtype,
                 void* workspace, size_t workspace_bytes, ofspmm_stream_t stream_) {
  return ofspmm_sddmm_ex(A, dY, B, dval, n, dense_dtype, nullptr, workspace, workspace_bytes, stream_);
}

int ofspmm_sddmm_ex(const ofspmm_csr* A, const void* dY, const void* B, void* dval, int64_t n, int dense_dtype,
                    const ofspmm_opts* opts, void* workspace, size_t workspace_bytes, ofspmm_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  // val_dtype is the dtype of the output dval here: a pattern matrix has no values to differentiate
  if (A != nullptr && unit(A)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  if (int rc = check_product(A, false, dense_dtype, n)) return rc;
  if (A->nnz == 0) return OFSPMM_OK;
  if (dval == nullptr) return OFSPMM_ERR_INVALID_ARG;
  const size_t val_size = A->val_dtype == OFSPMM_DTYPE_FLOAT ? 4 : 2;
  if (n == 0 || A->cols == 0) {
    OFSPMM_CUDA_OK(cudaMemsetAsync(dval, 0, static_cast<size_t>(A->nnz) * val_size, stream));
    return OFSPMM_OK;
  }
  if (dY == nullptr || B == nullptr) return OFSPMM_ERR_INVALID_ARG;
  const int64_t P = num_tasks(A->rows, A->nnz);
  const SddmmLayout L = sddmm_layout(A->rows, A->nnz);
  if (int rc = check_ws(workspace, workspace_bytes, L.total)) return rc;
  unsigned char* w = static_cast<unsigned char*>(workspace);
  const uint32_t fl = opts ? opts->flags : 0u;
  const bool dynamic = OFSPMM_DEFAULT_DYNAMIC_ORDER ? (fl & OFSPMM_ORDER_STATIC) == 0 : (fl & OFSPMM_ORDER_DYNAMIC) != 0;
  void* counter = dynamic ? w + L.counter : nullptr;
  // the SDDMM kernels use 256-item tasks: a plan of that task size is taken as is
  if (opts != nullptr && opts->plan != nullptr && opts->plan_bytes == plan_bytes_for(A->rows, A->nnz, kTaskItems))
    return launch_sddmm(A, dY, B, dval, n, dense_dtype, opts->plan, counter, P, stream);
  if (int rc = launch_task_partition(A->crow, A->idx_dtype, A->rows, A->nnz, P, kTaskItems, w + L.part, stream)) return rc;
  return launch_sddmm(A, dY, B, dval, n, dense_dtype, w + L.part, counter, P, stream);
}

int ofspmm_partition(const void* crow, int idx_dtype, int64_t rows, int64_t nnz, int64_t parts,
                     int64_t* out_row, int64_t* out_nz, ofspmm_stream_t stream) {
  if (crow == nullptr || out_row == nullptr || out_nz == nullptr) return OFSPMM_ERR_INVALID_ARG;
  if (rows < 0 || nnz < 0 || parts < 1) return OFSPMM_ERR_INVALID_ARG;
  if (!idx_ok(idx_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  return launch_partition_public(crow, idx_dtype, rows, nnz, parts, out_row, out_nz,
                                 reinterpret_cast<cudaStream_t>(stream));
}

int ofspmm_partition_host(const void* crow, int idx_dtype, int64_t rows, int64_t nnz, int64_t parts,
                          int64_t* out_row, int64_t* out_nz) {
  if (crow == nullptr || out_row == nullptr || out_nz == nullptr) return OFSPMM_ERR_INVALID_ARG;
  if (rows < 0 || nnz < 0 || parts < 1) return OFSPMM_ERR_INVALID_ARG;
  if (!idx_ok(idx_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  const int64_t total = rows + nnz;
  const int64_t ipw = (total + parts - 1) / parts;
  for (int64_t k = 0; k <= parts; ++k) {
    int64_t d = k * ipw;
    if (d > total) d = total;
    const int64_t r = idx_dtype == OFSPMM_DTYPE_INT32
                          ? merge_path_search<int32_t>(static_cast<const int32_t*>(crow), rows, nnz, d)
                          : merge_path_search<int64_t>(static_cast<const int64_t*>(crow), rows, nnz, d);
    out_row[k] = r;
    out_nz[k] = d - r;
  }
  return OFSPMM_OK;
}

int ofspmm_row_hist(const void* crow, int idx_dtype, int64_t rows, int64_t* hist32, ofspmm_stream_t stream) {
  if (crow == nullptr || hist32 == nullptr || rows < 0) return OFSPMM_ERR_INVALID_ARG;
  if (!idx_ok(idx_dtype)) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  return launch_row_hist(crow, idx_dtype, rows, hist32, reinterpret_cast<cudaStream_t>(stream));
}

size_t ofspmm_csr_transpose_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int idx_dtype) {
  if (rows < 0 || cols < 0 || nnz < 0 || !idx_ok(idx_dtype)) return 0;
  return transpose_workspace_bytes(rows, cols, nnz, idx_dtype);
}

int ofspmm_csr_transpose(const ofspmm_csr* A, void* t_crow, void* t_col, void* t_val, void* t_perm,
                         void* workspace, size_t workspace_bytes, ofspmm_stream_t stream) {
  if (int rc = check_csr(A, false)) return rc;
  if (t_crow == nullptr || (A->nnz > 0 && t_col == nullptr)) return OFSPMM_ERR_INVALID_ARG;
  if (unit(A) && t_val != nullptr) return OFSPMM_ERR_INVALID_ARG;  // a pattern A^T has no values
  return launch_transpose(A, t_crow, t_col, t_val, t_perm, workspace, workspace_bytes,
                          reinterpret_cast<cudaStream_t>(stream));
}

size_t ofspmm_fwd_host_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int64_t n, int dense_dtype,
                                       int idx_dtype, int val_dtype) {
  if (rows < 0 || cols < 0 || nnz < 0 || n < 0) return 0;
  return host_fwd_layout(rows, cols, nnz, n, dense_dtype, idx_dtype, val_dtype).total;
}

int ofspmm_fwd_host(const ofspmm_csr* Ah, const void* B_host, void* C_host, int64_t n, int dense_dtype,
                    void* workspace, size_t workspace_bytes, ofspmm_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (int rc = check_fwd(Ah, B_host, C_host, n, dense_dtype)) return rc;
  if (Ah->rows == 0 || n == 0) return OFSPMM_OK;
  const HostFwdLayout L = host_fwd_layout(Ah->rows, Ah->cols, Ah->nnz, n, dense_dtype, Ah->idx_dtype, Ah->val_dtype);
  if (int rc = check_ws(workspace, workspace_bytes, L.total)) return rc;
  const size_t is = idx_size(Ah->idx_dtype), vs = val_size(Ah->val_dtype);
  const size_t ds = dense_size(dense_dtype);
  unsigned char* w = static_cast<unsigned char*>(workspace);
  OFSPMM_CUDA_OK(cudaMemcpyAsync(w + L.crow, Ah->crow, static_cast<size_t>(Ah->rows + 1) * is, cudaMemcpyHostToDevice, stream));
  if (Ah->nnz > 0) {
    OFSPMM_CUDA_OK(cudaMemcpyAsync(w + L.col, Ah->col, static_cast<size_t>(Ah->nnz) * is, cudaMemcpyHostToDevice, stream));
    if (!unit(Ah))
      OFSPMM_CUDA_OK(cudaMemcpyAsync(w + L.val, Ah->val, static_cast<size_t>(Ah->nnz) * vs, cudaMemcpyHostToDevice, stream));
  }
  if (Ah->cols > 0 && B_host != nullptr)
    OFSPMM_CUDA_OK(cudaMemcpyAsync(w + L.B, B_host, static_cast<size_t>(Ah->cols) * n * ds, cudaMemcpyHostToDevice, stream));
  ofspmm_csr Ad = *Ah;
  Ad.crow = w + L.crow;
  Ad.col = w + L.col;
  Ad.val = unit(Ah) ? nullptr : w + L.val;
  if (int rc = run_fwd(&Ad, w + L.B, n, w + L.C, n, n, dense_dtype, nullptr, w + L.fws, workspace_bytes - L.fws, stream)) return rc;
  OFSPMM_CUDA_OK(cudaMemcpyAsync(C_host, w + L.C, static_cast<size_t>(Ah->rows) * n * ds, cudaMemcpyDeviceToHost, stream));
  return OFSPMM_OK;
}

const char* ofspmm_strerror(int status) {
  switch (status) {
    case OFSPMM_OK: return "ok";
    case OFSPMM_ERR_INVALID_ARG: return "invalid argument (null pointer, negative size or inconsistent shape)";
    case OFSPMM_ERR_UNSUPPORTED_DTYPE: return "unsupported dtype combination";
    case OFSPMM_ERR_WORKSPACE: return "workspace missing, misaligned or smaller than *_workspace_bytes()";
    case OFSPMM_ERR_CUDA: return "CUDA runtime call or kernel launch failed";
    case OFSPMM_ERR_TOO_LARGE: return "rows >= 2^31-1, or nnz >= 2^31-1 with int32 indices";
    case OFSPMM_ERR_NO_DEVICE: return "no sm_100 (B200) device current on this thread";
    default: return "unknown status";
  }
}

int ofspmm_version(void) { return 100; }

uint64_t ofspmm_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

const char* ofspmm_fwd_variant(int64_t rows, int64_t nnz, int64_t n, int dense_dtype) {
  return ofspmm_variant_name(OFSPMM_VARIANT_AUTO, rows, nnz, n, dense_dtype);
}

const char* ofspmm_variant_name(int variant, int64_t rows, int64_t nnz, int64_t n, int dense_dtype) {
  // "<schedule family>/<lane layout>": family from the variant, layout from the dense width
  static thread_local char buf[160];
  const FwdVariant v = resolve_variant(variant, rows, nnz, n, dense_dtype);
  const char* fam = v.whole_rows               ? "whole_rows(one launch, no merge path)"
                    : v.items == kSmallTaskItems ? "merge_path(64-item tasks)"
                    : v.row_parallel           ? "merge_path(256-item tasks, row-parallel groups)"
                                               : "merge_path(256-item tasks)";
  if (v.whole_rows) {
    snprintf(buf, sizeof(buf), "%s/group-per-row(%d lanes x 16B, 4 gathers in flight)", fam,
             lane_layout(LaneOp::kFwdRows, dense_dtype, n, true).lpr);
    return buf;
  }
  snprintf(buf, sizeof(buf), "%s/%s", fam, fwd_variant_name(n, dense_dtype, true));
  return buf;
}

}  // extern "C"
