// fwd.cu — variant resolution and dispatch of the merge-path SpMM forward to its kernel family
// (fwd_launch.cuh), plus the task partitioner launch.
#include "launch.cuh"
#include "spmm_kernels.cuh"

namespace ofspmm {

int launch_family_base(const FwdParams&, const LaneLayout&, int, int, int, const FwdLaunch&, cudaStream_t);
int launch_family_small(const FwdParams&, const LaneLayout&, int, int, int, const FwdLaunch&, cudaStream_t);
int launch_family_rowpar(const FwdParams&, const LaneLayout&, int, int, int, const FwdLaunch&, cudaStream_t);
int launch_family_rows(const FwdParams&, const LaneLayout&, int, int, cudaStream_t);

namespace {

// B, C and the bias allow 16-byte vector rows: aligned addresses, strides a whole number of vectors.
bool vec_rows_ok(const void* B, int64_t ldb, const void* C, int64_t ldc, int dense_dtype, const FwdLaunch& L) {
  const int64_t v = dense_vec_width(dense_dtype);
  const uintptr_t bits = reinterpret_cast<uintptr_t>(B) | reinterpret_cast<uintptr_t>(C) |
                         ((L.flags & kFwdBias) ? reinterpret_cast<uintptr_t>(L.bias) : 0);
  return (bits & 15) == 0 && ldb % v == 0 && ldc % v == 0;
}

}  // namespace

// AUTO (no histogram available): decided from the host-known sizes only — fewer 256-item tasks
// than resident warps -> 64-item tasks.  With the row-length histogram on the host,
// ofspmm_choose_variant() may also pick the row-parallel layout (api.cu).
// Wide matrices (wide_nnz) have 256-item merge-path kernels only: an explicit whole-row or
// 64-item code falls back to them (AUTO never picks 64-item tasks at that size anyway).
// The row-parallel and whole-row layouts are looked up for 16-byte aligned rows; a launch whose
// rows are not falls back to another family.
FwdVariant resolve_variant(int variant, int64_t rows, int64_t nnz, int64_t n, int dense_dtype) {
  const bool rowpar_supported = lane_layout(LaneOp::kFwdRowPar, dense_dtype, n, true).ok();
  FwdVariant v{kTaskItems, false, false};
  if (wide_nnz(nnz)) {
    v.row_parallel = (variant & OFSPMM_VARIANT_EXPLICIT) && (variant & OFSPMM_VARIANT_ROWPAR) &&
                     !(variant & (OFSPMM_VARIANT_ROWS | OFSPMM_VARIANT_ITEMS64)) && rowpar_supported;
    return v;
  }
  if (variant & OFSPMM_VARIANT_EXPLICIT) {
    if (variant & OFSPMM_VARIANT_ROWS) {
      // sized like the 64-item family, which is also what runs when a launch cannot use the
      // whole-row kernel (int64 indices, unaligned or strided-odd rows)
      v.items = kSmallTaskItems;
      v.whole_rows = lane_layout(LaneOp::kFwdRows, dense_dtype, n, true).ok();
    } else if (variant & OFSPMM_VARIANT_ITEMS64) v.items = kSmallTaskItems;
    else if ((variant & OFSPMM_VARIANT_ROWPAR) && rowpar_supported) v.row_parallel = true;
    return v;
  }
  if (num_tasks(rows, nnz, kTaskItems) < kSmallProblemTasks) v.items = kSmallTaskItems;
  return v;
}

int encode_variant(const FwdVariant& v) {
  int code = OFSPMM_VARIANT_EXPLICIT;
  if (v.whole_rows) code |= OFSPMM_VARIANT_ROWS;
  else if (v.items == kSmallTaskItems) code |= OFSPMM_VARIANT_ITEMS64;
  if (v.row_parallel) code |= OFSPMM_VARIANT_ROWPAR;
  return code;
}

int launch_task_partition(const void* crow, int idx_dtype, int64_t rows, int64_t nnz, int64_t P,
                          int items, void* part, cudaStream_t stream) {
  const int threads = 256;
  const unsigned blocks = static_cast<unsigned>((P + 1 + threads - 1) / threads);
  return dispatch_index<true>(idx_dtype, wide_nnz(nnz), [&](auto idx, auto pt) {
    using IdxT = typename decltype(idx)::type;
    using PartT = typename decltype(pt)::type;
    task_partition_kernel<IdxT, PartT><<<blocks, threads, 0, stream>>>(
        static_cast<const IdxT*>(crow), static_cast<int>(rows), static_cast<typename PartOf<PartT>::Nz>(nnz), items,
        static_cast<int>(P), static_cast<PartT*>(part));
    return launched();
  });
}

// The whole-row kernel needs what resolve_variant cannot see: the pointers' alignment, the
// strides and the index dtype of THIS call.  It never serves a wide matrix (resolve_variant
// clears whole_rows for those; they have int64 indices besides).
bool rows_kernel_applies(const ofspmm_csr* A, const void* B, int64_t ldb, const void* C, int64_t ldc, int64_t n,
                         int dense_dtype, const FwdLaunch& L) {
  return L.variant.whole_rows && A->idx_dtype == OFSPMM_DTYPE_INT32 &&
         lane_layout(LaneOp::kFwdRows, dense_dtype, n, vec_rows_ok(B, ldb, C, ldc, dense_dtype, L)).ok();
}

int launch_fwd(const ofspmm_csr* A, const void* B, int64_t ldb, void* C, int64_t ldc, int64_t n,
               int dense_dtype, const void* part, float* carry, float* head, void* counter, int64_t P,
               const FwdLaunch& L, cudaStream_t stream) {
  FwdParams p;
  p.ldb = ldb;
  p.ldc = ldc;
  p.crow = A->crow;
  p.col = A->col;
  p.val = A->val;
  p.B = B;
  p.C = C;
  p.part = part;
  p.carry = carry;
  p.head = head;
  p.cols = A->cols;
  p.rows = static_cast<int>(A->rows);
  p.n = static_cast<int>(n);
  p.P = static_cast<int>(P);
  p.panels = 1;
  p.bias = L.bias;
  p.flags = L.flags;
  p.acc32 = L.acc32;
  p.counter = L.dynamic ? static_cast<unsigned int*>(counter) : nullptr;
  if (rows_kernel_applies(A, B, ldb, C, ldc, n, dense_dtype, L)) {
    p.counter = nullptr;
    return launch_family_rows(p, lane_layout(LaneOp::kFwdRows, dense_dtype, n, true), dense_dtype, A->val_dtype, stream);
  }
  const bool vec_rows = vec_rows_ok(B, ldb, C, ldc, dense_dtype, L);
  if (L.variant.row_parallel) {  // 256-item tasks only (resolve_variant)
    const LaneLayout rowpar = lane_layout(LaneOp::kFwdRowPar, dense_dtype, n, vec_rows);
    if (rowpar.ok()) return launch_family_rowpar(p, rowpar, A->idx_dtype, dense_dtype, A->val_dtype, L, stream);
  }
  const LaneLayout l = lane_layout(LaneOp::kFwd, dense_dtype, n, vec_rows);
  if (L.variant.items == kSmallTaskItems) return launch_family_small(p, l, A->idx_dtype, dense_dtype, A->val_dtype, L, stream);
  return launch_family_base(p, l, A->idx_dtype, dense_dtype, A->val_dtype, L, stream);
}

const char* fwd_variant_name(int64_t n, int dense_dtype, bool aligned) {
  const LaneLayout l = lane_layout(LaneOp::kFwd, dense_dtype, n, aligned);
  if (l.vec == 1) return "warp-per-row(scalar lanes, unaligned n)";
  if (l.lpr == 8) return "vector-per-row(8 lanes x 16B, 4 nnz per step)";
  if (l.lpr == 16) return "vector-per-row(16 lanes x 16B, 2 nnz per step)";
  if (l.ch == 1) return "warp-per-row(32 lanes x 16B)";
  if (l.ch == 2) return "warp-per-row(32 lanes x 2 x 16B)";
  return "warp-per-row(32 lanes x 4 x 16B, column panels)";
}

}  // namespace ofspmm
