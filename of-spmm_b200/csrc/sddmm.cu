// sddmm.cu — variant selection and launch of the SDDMM value-gradient kernels.
#include "launch.cuh"
#include "sddmm_bwd_kernels.cuh"

namespace ofspmm {

namespace {

template <typename Stage, typename Kern>
int launch_persistent(Kern kern, SddmmParams p, bool dynamic_ok, KernelLaunchCache& cache, cudaStream_t stream) {
  constexpr int WARPS = kWarpsPerCta;
  constexpr size_t smem = kMergeSmem<Stage>;
  int sms = 0, occ = 0;
  if (int rc = merge_residency(kern, smem, cache, &sms, &occ)) return rc;
  const int64_t ctas_needed = (static_cast<int64_t>(p.P) + WARPS - 1) / WARPS;
  const int64_t resident = static_cast<int64_t>(sms) * occ;
  const int gx = static_cast<int>(ctas_needed < resident ? ctas_needed : resident);
  if (!dynamic_ok || gx == ctas_needed) p.counter = nullptr;
  if (p.counter != nullptr) OFSPMM_CUDA_OK(cudaMemsetAsync(p.counter, 0, sizeof(unsigned int), stream));
  kern<<<gx, WARPS * 32, smem, stream>>>(p);
  count_launch();
  OFSPMM_CUDA_OK(cudaGetLastError());
  return OFSPMM_OK;
}

// The layouts lane_layout can pick for the SDDMM; no layout (rows wider than the register tile):
// sddmm_wide_kernel, which loops over the row.
template <typename DT, typename ValT, typename IdxT, typename PartT>
int launch_typed(const SddmmParams& p, const LaneLayout& l, cudaStream_t stream) {
  constexpr int ITEMS = kTaskItems;
  constexpr int WARPS = kWarpsPerCta;
  using Stage = TaskStage<IdxT, float, ITEMS>;
  constexpr int V = vec_width(sizeof(DT));
  return dispatch_lanes<Lanes<V, 8, 1>, Lanes<V, 16, 1>, Lanes<V, 32, 1>, Lanes<V, 32, 2>, Lanes<V, 32, 4>, Lanes<V, 0, 0>,
                        Lanes<1, 32, 1>, Lanes<1, 32, 4>, Lanes<1, 0, 0>>(l, [&](auto lanes) {
    using S = decltype(lanes);
    if constexpr (S::LPR == 0) {
      static KernelLaunchCache cache;
      return launch_persistent<Stage>(sddmm_wide_kernel<DT, ValT, IdxT, S::VEC, ITEMS, WARPS, PartT>, p, false, cache, stream);
    } else {
      static KernelLaunchCache cache_full, cache_masked;
      if (l.full)
        return launch_persistent<Stage>(sddmm_merge_kernel<DT, ValT, IdxT, S::VEC, S::LPR, S::CH, true, ITEMS, WARPS, PartT>,
                                        p, true, cache_full, stream);
      return launch_persistent<Stage>(sddmm_merge_kernel<DT, ValT, IdxT, S::VEC, S::LPR, S::CH, false, ITEMS, WARPS, PartT>,
                                      p, true, cache_masked, stream);
    }
  });
}

}  // namespace

int launch_sddmm(const ofspmm_csr* A, const void* dY, const void* B, void* dval, int64_t n,
                 int dense_dtype, const void* part, void* counter, int64_t P, cudaStream_t stream) {
  SddmmParams p;
  p.counter = static_cast<unsigned int*>(counter);
  p.crow = A->crow;
  p.col = A->col;
  p.dY = dY;
  p.B = B;
  p.dval = dval;
  p.part = part;
  p.cols = A->cols;
  p.rows = static_cast<int>(A->rows);
  p.n = static_cast<int>(n);
  p.P = static_cast<int>(P);
  const bool aligned = ((reinterpret_cast<uintptr_t>(B) | reinterpret_cast<uintptr_t>(dY)) & 15) == 0;
  const LaneLayout l = lane_layout(LaneOp::kSddmm, dense_dtype, n, aligned);
  return dispatch_index<true>(A->idx_dtype, wide_nnz(A->nnz), [&](auto idx, auto part) {
    return dispatch_dtypes<false>(dense_dtype, A->val_dtype, [&](auto dense, auto val) {  // dval has a dtype
      return launch_typed<typename decltype(dense)::type, typename decltype(val)::type, typename decltype(idx)::type,
                          typename decltype(part)::type>(p, l, stream);
    });
  });
}

}  // namespace ofspmm
