// launch.cuh — host-side dispatch shared by the launchers of the merge-path kernels (fwd_launch.cuh,
// fwd_rows.cu, sddmm.cu, bwd.cu): runtime dtype codes and lane layouts to template arguments, and
// the launch constants of a kernel on the current device.
#pragma once
#include "common.cuh"
#include "internal.h"

namespace ofspmm {

template <typename T>
struct Tag { using type = T; };

// f(Tag<DT>{}, Tag<ValT>{}) for a (dense, value) dtype pair; kUnit: the caller has kernels for
// pattern matrices (UnitVal) too.
template <bool kUnit, typename F>
int dispatch_dtypes(int dense_dtype, int val_dtype, F&& f) {
  const bool f32 = dense_dtype == OFSPMM_DTYPE_FLOAT, bf16 = dense_dtype == OFSPMM_DTYPE_BFLOAT16;
  if (f32 && val_dtype == OFSPMM_DTYPE_FLOAT) return f(Tag<float>{}, Tag<float>{});
  if (bf16 && val_dtype == OFSPMM_DTYPE_FLOAT) return f(Tag<__nv_bfloat16>{}, Tag<float>{});
  if (bf16 && val_dtype == OFSPMM_DTYPE_BFLOAT16) return f(Tag<__nv_bfloat16>{}, Tag<__nv_bfloat16>{});
  if constexpr (kUnit) {
    if (f32 && val_dtype == OFSPMM_VAL_UNIT) return f(Tag<float>{}, Tag<UnitVal>{});
    if (bf16 && val_dtype == OFSPMM_VAL_UNIT) return f(Tag<__nv_bfloat16>{}, Tag<UnitVal>{});
  }
  return OFSPMM_ERR_UNSUPPORTED_DTYPE;
}

// f(Tag<IdxT>{}, Tag<PartT>{}) for the index dtype.  A wide matrix (wide_nnz: int64 indices) takes
// 16-byte partition entries, where the caller has such kernels (kWide); otherwise TOO_LARGE.
template <bool kWide, typename F>
int dispatch_index(int idx_dtype, bool wide, F&& f) {
  if (!wide) {
    if (idx_dtype == OFSPMM_DTYPE_INT32) return f(Tag<int32_t>{}, Tag<int2>{});
    if (idx_dtype == OFSPMM_DTYPE_INT64) return f(Tag<int64_t>{}, Tag<int2>{});
  } else if constexpr (kWide) {
    if (idx_dtype == OFSPMM_DTYPE_INT64) return f(Tag<int64_t>{}, Tag<longlong2>{});
  }
  return wide ? OFSPMM_ERR_TOO_LARGE : OFSPMM_ERR_UNSUPPORTED_DTYPE;
}

template <int V, int L, int C>
struct Lanes { static constexpr int VEC = V, LPR = L, CH = C; };

// f(Ls{}) for the one of the caller's instantiated layouts `Ls` that `l` names (Lanes<VEC, 0, 0>:
// the "no layout" answer of lane_layout); INVALID_ARG if none does.
template <typename... Ls, typename F>
int dispatch_lanes(const LaneLayout& l, F&& f) {
  int rc = OFSPMM_ERR_INVALID_ARG;
  (void)((l.vec == Ls::VEC && l.lpr == Ls::LPR && l.ch == Ls::CH && ((rc = f(Ls{})), true)) || ...);
  return rc;
}

// Dynamic shared memory of a merge-path kernel: one task stage and one mbarrier per warp.
template <typename Stage>
constexpr size_t kMergeSmem = (sizeof(Stage) + sizeof(uint64_t)) * kWarpsPerCta;

// SM count of the current device and resident CTAs per SM of `kern` with `smem` bytes of dynamic
// shared memory.  The smem opt-in and the occupancy are immutable facts of the binary and device,
// set and queried once per (kernel, device) in `cache`: that only removes ~5 us of driver calls
// from every launch, it is not mutable state in the sense of SURVEY.md §8b.
template <typename Kern>
int merge_residency(Kern kern, size_t smem, KernelLaunchCache& cache, int* sms, int* occ) {
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  *sms = dev.sms;
  *occ = cache.get(dev.ordinal);
  if (*occ == 0) {
    OFSPMM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    OFSPMM_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, kern, kWarpsPerCta * 32, smem));
    if (*occ < 1) return OFSPMM_ERR_CUDA;
    cache.set(dev.ordinal, *occ);
  }
  return OFSPMM_OK;
}

}  // namespace ofspmm
