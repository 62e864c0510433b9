// fwd_launch.cuh — launch of one *family* of merge-path SpMM kernels.  A family fixes the
// compile-time schedule knobs (merge items per task, nnz- vs row-parallel lane layout); inside a
// family the lane layout follows the dense width and dtype.  Each family is instantiated in its
// own translation unit (fwd_base.cu, fwd_small.cu, fwd_extra.cu) so the library builds in
// parallel; fwd.cu picks the family from the variant (internal.h:FwdVariant).
#pragma once
#include "internal.h"
#include "spmm_kernels.cuh"

namespace ofspmm {

template <typename DT, typename ValT, typename IdxT, typename PartT, int VEC, int LPR, int CH, bool kFull, bool kRowPar, int ITEMS>
int launch_full(FwdParams p, int panels, const FwdLaunch& L, cudaStream_t stream) {
  if (static_cast<int64_t>(p.P) * panels >= kMaxTasks) return OFSPMM_ERR_TOO_LARGE;
  p.panels = panels;
  constexpr int WARPS = kWarpsPerCta;
  auto kern = spmm_merge_kernel<DT, ValT, IdxT, VEC, LPR, CH, kFull, kRowPar, ITEMS, WARPS, PartT>;
  const size_t smem = sizeof(TaskStage<IdxT, ValT, ITEMS>) * WARPS + sizeof(uint64_t) * WARPS;
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  // per (kernel, device) launch constants, queried once: the shared-memory opt-in and the
  // occupancy are immutable facts of the binary + device, so memoising them is not mutable state
  // in the sense of SURVEY.md §8b — it only removes ~5 us of driver calls from every launch
  static KernelLaunchCache cache;
  int occ = cache.get(dev.ordinal);
  if (occ == 0) {
    OFSPMM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    OFSPMM_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, WARPS * 32, smem));
    if (occ < 1) return OFSPMM_ERR_CUDA;
    cache.set(dev.ordinal, occ);
  }
  // persistent grid: a whole number of CTAs per SM (148 SMs on B200), never more than the tasks
  const int64_t ctas_needed = (static_cast<int64_t>(p.P) + WARPS - 1) / WARPS;
  const int64_t ctas_all = (static_cast<int64_t>(p.P) * panels + WARPS - 1) / WARPS;
  // reserve_ctas: leave that many CTA slots per SM to the exchange kernels of the multi-GPU path
  const int occ_used = L.reserve_ctas > 0 ? (occ - L.reserve_ctas > 1 ? occ - L.reserve_ctas : 1) : occ;
  const int64_t resident = static_cast<int64_t>(dev.sms) * occ_used;
  int64_t gx64 = ctas_all < resident ? ctas_all : resident;
  // tasks_per_warp = k > 0 (ofspmm_opts): a non-persistent grid whose CTAs retire after k tasks
  // per warp, so kernels of another stream (NCCL collectives, the peer-pull kernel of the
  // multi-GPU path) get SMs while this kernel is still running.
  p.max_tasks = 0;
  if (L.tasks_per_warp > 0) {
    const int64_t want = (ctas_all + L.tasks_per_warp - 1) / L.tasks_per_warp;
    if (want > gx64) {
      gx64 = want;
      p.max_tasks = L.tasks_per_warp;  // gx64 * WARPS * max_tasks >= tasks: every task gets drawn
    }
  }
  if (gx64 == ctas_all) p.counter = nullptr;  // one task per warp: nothing to draw
  if (p.counter != nullptr) OFSPMM_CUDA_OK(cudaMemsetAsync(p.counter, 0, sizeof(unsigned int), stream));
  const int gx = static_cast<int>(gx64);
  kern<<<gx, WARPS * 32, smem, stream>>>(p);
  count_launch();
  OFSPMM_CUDA_OK(cudaGetLastError());
  if (p.P > 1) {  // stitch rows that span several tasks (a single task cannot split a row)
    auto fix = spmm_fixup_kernel<DT, IdxT, VEC, WARPS, PartT>;
    fix<<<static_cast<unsigned>((ctas_needed + 31) / 32), WARPS * 32, 0, stream>>>(p);  // one lane per task
    count_launch();
    OFSPMM_CUDA_OK(cudaGetLastError());
  }
  return OFSPMM_OK;
}

// kFull (no masked lanes, immediate chunk offsets) when n is a whole number of register tiles.
template <typename DT, typename ValT, typename IdxT, typename PartT, int VEC, int LPR, int CH, bool kRowPar, int ITEMS>
int launch_one(const FwdParams& p, int panels, const FwdLaunch& L, cudaStream_t stream) {
  if (p.n % (LPR * VEC * CH) == 0)
    return launch_full<DT, ValT, IdxT, PartT, VEC, LPR, CH, true, kRowPar, ITEMS>(p, panels, L, stream);
  return launch_full<DT, ValT, IdxT, PartT, VEC, LPR, CH, false, kRowPar, ITEMS>(p, panels, L, stream);
}

// Lane layout by dense width: 8 / 16 lanes per row (vector-per-row: 4 / 2 non-zero groups per
// warp instruction) or 32 lanes x 1 / 2 / 4 16-byte chunks (warp-per-row); scalar lanes when the
// rows are not 16-byte aligned.  The row-parallel family only exists for the sub-warp layouts
// (fwd.cu checks rowpar_supported() first).
template <typename DT, typename ValT, typename IdxT, typename PartT, bool kRowPar, int ITEMS>
int launch_typed(const FwdParams& p, bool aligned, const FwdLaunch& L, cudaStream_t stream) {
  constexpr int VECW = 16 / sizeof(DT);
  const int n = p.n;
  if (aligned && n % VECW == 0 && p.ldb % VECW == 0 && p.ldc % VECW == 0) {
    const int nvec = n / VECW;
    if (nvec <= 8) return launch_one<DT, ValT, IdxT, PartT, VECW, 8, 1, kRowPar, ITEMS>(p, 1, L, stream);
    if (nvec <= 16) return launch_one<DT, ValT, IdxT, PartT, VECW, 16, 1, kRowPar, ITEMS>(p, 1, L, stream);
    if constexpr (!kRowPar) {
      if (nvec <= 32) return launch_one<DT, ValT, IdxT, PartT, VECW, 32, 1, false, ITEMS>(p, 1, L, stream);
      if (nvec <= 64) return launch_one<DT, ValT, IdxT, PartT, VECW, 32, 2, false, ITEMS>(p, 1, L, stream);
      return launch_one<DT, ValT, IdxT, PartT, VECW, 32, 4, false, ITEMS>(p, (nvec + 127) / 128, L, stream);
    }
    return OFSPMM_ERR_INVALID_ARG;  // unreachable: rowpar_supported() guards it
  }
  if constexpr (!kRowPar) {
    if (n <= 32) return launch_one<DT, ValT, IdxT, PartT, 1, 32, 1, false, ITEMS>(p, 1, L, stream);
    if (n <= 64) return launch_one<DT, ValT, IdxT, PartT, 1, 32, 2, false, ITEMS>(p, 1, L, stream);
    if (n <= 128) return launch_one<DT, ValT, IdxT, PartT, 1, 32, 4, false, ITEMS>(p, 1, L, stream);
    return launch_one<DT, ValT, IdxT, PartT, 1, 32, 8, false, ITEMS>(p, (n + 255) / 256, L, stream);
  }
  return OFSPMM_ERR_INVALID_ARG;
}

template <typename IdxT, typename PartT, bool kRowPar, int ITEMS>
int launch_idx(const FwdParams& p, int dense_dtype, int val_dtype, bool aligned, const FwdLaunch& L,
               cudaStream_t stream) {
  if (dense_dtype == OFSPMM_DTYPE_FLOAT && val_dtype == OFSPMM_DTYPE_FLOAT)
    return launch_typed<float, float, IdxT, PartT, kRowPar, ITEMS>(p, aligned, L, stream);
  if (dense_dtype == OFSPMM_DTYPE_BFLOAT16 && val_dtype == OFSPMM_DTYPE_FLOAT)
    return launch_typed<__nv_bfloat16, float, IdxT, PartT, kRowPar, ITEMS>(p, aligned, L, stream);
  if (dense_dtype == OFSPMM_DTYPE_BFLOAT16 && val_dtype == OFSPMM_DTYPE_BFLOAT16)
    return launch_typed<__nv_bfloat16, __nv_bfloat16, IdxT, PartT, kRowPar, ITEMS>(p, aligned, L, stream);
  if (dense_dtype == OFSPMM_DTYPE_FLOAT && val_dtype == OFSPMM_VAL_UNIT)
    return launch_typed<float, UnitVal, IdxT, PartT, kRowPar, ITEMS>(p, aligned, L, stream);
  if (dense_dtype == OFSPMM_DTYPE_BFLOAT16 && val_dtype == OFSPMM_VAL_UNIT)
    return launch_typed<__nv_bfloat16, UnitVal, IdxT, PartT, kRowPar, ITEMS>(p, aligned, L, stream);
  return OFSPMM_ERR_UNSUPPORTED_DTYPE;
}

template <bool kRowPar, int ITEMS>
int launch_family(const FwdParams& p, int idx_dtype, int dense_dtype, int val_dtype, bool aligned,
                  const FwdLaunch& L, cudaStream_t stream) {
  if (idx_dtype == OFSPMM_DTYPE_INT32 && !L.wide)
    return launch_idx<int32_t, int2, kRowPar, ITEMS>(p, dense_dtype, val_dtype, aligned, L, stream);
  if (idx_dtype == OFSPMM_DTYPE_INT64 && !L.wide)
    return launch_idx<int64_t, int2, kRowPar, ITEMS>(p, dense_dtype, val_dtype, aligned, L, stream);
  // wide matrices: 256-item tasks only (resolve_variant never gives them 64-item tasks)
  if constexpr (ITEMS == kTaskItems) {
    if (idx_dtype == OFSPMM_DTYPE_INT64) return launch_idx<int64_t, longlong2, kRowPar, ITEMS>(p, dense_dtype, val_dtype, aligned, L, stream);
  }
  return L.wide ? OFSPMM_ERR_TOO_LARGE : OFSPMM_ERR_UNSUPPORTED_DTYPE;
}

}  // namespace ofspmm
