// fwd_launch.cuh — launch of one *family* of merge-path SpMM kernels.  A family fixes the
// compile-time schedule knobs (merge items per task, nnz- vs row-parallel lane layout); inside a
// family the lane layout follows the dense width and dtype.  Each family is instantiated in its
// own translation unit (fwd_base.cu, fwd_small.cu, fwd_extra.cu) so the library builds in
// parallel; fwd.cu picks the family from the variant (internal.h:FwdVariant).
#pragma once
#include "launch.cuh"
#include "spmm_kernels.cuh"

namespace ofspmm {

template <typename DT, typename ValT, typename IdxT, typename PartT, int VEC, int LPR, int CH, bool kFull, bool kRowPar, int ITEMS>
int launch_full(FwdParams p, int panels, const FwdLaunch& L, cudaStream_t stream) {
  if (static_cast<int64_t>(p.P) * panels >= kMaxTasks) return OFSPMM_ERR_TOO_LARGE;
  p.panels = panels;
  constexpr int WARPS = kWarpsPerCta;
  auto kern = spmm_merge_kernel<DT, ValT, IdxT, VEC, LPR, CH, kFull, kRowPar, ITEMS, WARPS, PartT>;
  constexpr size_t smem = kMergeSmem<TaskStage<IdxT, ValT, ITEMS>>;
  static KernelLaunchCache cache;
  int sms = 0, occ = 0;
  if (int rc = merge_residency(kern, smem, cache, &sms, &occ)) return rc;
  // persistent grid: a whole number of CTAs per SM (148 SMs on B200), never more than the tasks
  const int64_t ctas_needed = (static_cast<int64_t>(p.P) + WARPS - 1) / WARPS;
  const int64_t ctas_all = (static_cast<int64_t>(p.P) * panels + WARPS - 1) / WARPS;
  // reserve_ctas: leave that many CTA slots per SM to the exchange kernels of the multi-GPU path
  const int occ_used = L.reserve_ctas > 0 ? (occ - L.reserve_ctas > 1 ? occ - L.reserve_ctas : 1) : occ;
  const int64_t resident = static_cast<int64_t>(sms) * occ_used;
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

// The layouts each family instantiates (lane_layout picks one): 8 / 16 lanes per row
// (vector-per-row: 4 / 2 non-zero groups per warp instruction) or 32 lanes x 1 / 2 / 4 16-byte
// chunks (warp-per-row); scalar lanes when the rows are not 16-byte aligned.  The row-parallel
// family only has the sub-warp layouts.  kFull (no masked lanes, immediate chunk offsets) when n is
// a whole number of register tiles.
template <typename DT, typename ValT, typename IdxT, typename PartT, bool kRowPar, int ITEMS>
int launch_typed(const FwdParams& p, const LaneLayout& l, const FwdLaunch& L, cudaStream_t stream) {
  constexpr int V = vec_width(sizeof(DT));
  auto go = [&](auto lanes) {
    using S = decltype(lanes);
    if (l.full) return launch_full<DT, ValT, IdxT, PartT, S::VEC, S::LPR, S::CH, true, kRowPar, ITEMS>(p, l.panels, L, stream);
    return launch_full<DT, ValT, IdxT, PartT, S::VEC, S::LPR, S::CH, false, kRowPar, ITEMS>(p, l.panels, L, stream);
  };
  if constexpr (kRowPar) {
    return dispatch_lanes<Lanes<V, 8, 1>, Lanes<V, 16, 1>>(l, go);
  } else {
    return dispatch_lanes<Lanes<V, 8, 1>, Lanes<V, 16, 1>, Lanes<V, 32, 1>, Lanes<V, 32, 2>, Lanes<V, 32, 4>,
                          Lanes<1, 32, 1>, Lanes<1, 32, 2>, Lanes<1, 32, 4>, Lanes<1, 32, 8>>(l, go);
  }
}

// Wide matrices have 256-item tasks only (resolve_variant never gives them 64-item tasks).
template <bool kRowPar, int ITEMS>
int launch_family(const FwdParams& p, const LaneLayout& l, int idx_dtype, int dense_dtype, int val_dtype,
                  const FwdLaunch& L, cudaStream_t stream) {
  return dispatch_index<ITEMS == kTaskItems>(idx_dtype, L.wide, [&](auto idx, auto part) {
    return dispatch_dtypes<true>(dense_dtype, val_dtype, [&](auto dense, auto val) {
      return launch_typed<typename decltype(dense)::type, typename decltype(val)::type, typename decltype(idx)::type,
                          typename decltype(part)::type, kRowPar, ITEMS>(p, l, L, stream);
    });
  });
}

}  // namespace ofspmm
