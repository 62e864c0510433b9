// bwd.cu — launch of the atomic A^T·dY scatter (route 2 of ofspmm_bwd_b).
#include "launch.cuh"
#include "sddmm_bwd_kernels.cuh"

namespace ofspmm {

namespace {

template <typename DT, typename ValT, typename IdxT, typename PartT, int VEC, int LPR, int CH>
int launch_one(const BwdAtomicParams& p, int panels, cudaStream_t stream) {
  constexpr int ITEMS = kTaskItems;
  constexpr int WARPS = kWarpsPerCta;
  auto kern = bwd_atomic_kernel<DT, ValT, IdxT, VEC, LPR, CH, ITEMS, WARPS, PartT>;
  constexpr size_t smem = kMergeSmem<TaskStage<IdxT, ValT, ITEMS>>;
  static KernelLaunchCache cache;
  int sms = 0, occ = 0;
  if (int rc = merge_residency(kern, smem, cache, &sms, &occ)) return rc;
  // 2-D grid: the column panels side by side, each with at least one CTA per SM
  const int64_t ctas_needed = (static_cast<int64_t>(p.P) + WARPS - 1) / WARPS;
  int64_t per_panel = static_cast<int64_t>(sms) * occ / panels;
  if (per_panel < sms) per_panel = sms;
  const int gx = static_cast<int>(ctas_needed < per_panel ? ctas_needed : per_panel);
  kern<<<dim3(gx, panels), WARPS * 32, smem, stream>>>(p);
  count_launch();
  OFSPMM_CUDA_OK(cudaGetLastError());
  return OFSPMM_OK;
}

// The layouts lane_layout can pick for the atomic scatter.
template <typename DT, typename ValT, typename IdxT, typename PartT>
int launch_typed(const BwdAtomicParams& p, const LaneLayout& l, cudaStream_t stream) {
  constexpr int V = vec_width(sizeof(DT));
  return dispatch_lanes<Lanes<V, 8, 1>, Lanes<V, 16, 1>, Lanes<V, 32, 1>, Lanes<V, 32, 2>, Lanes<V, 32, 4>,
                        Lanes<1, 32, 1>, Lanes<1, 32, 4>, Lanes<1, 32, 8>>(l, [&](auto lanes) {
    using S = decltype(lanes);
    return launch_one<DT, ValT, IdxT, PartT, S::VEC, S::LPR, S::CH>(p, l.panels, stream);
  });
}

}  // namespace

int launch_bwd_atomic(const ofspmm_csr* A, const void* dY, float* acc, void* dB_cast_out, int64_t n,
                      int dense_dtype, const void* part, int64_t P, cudaStream_t stream) {
  const size_t out_elems = static_cast<size_t>(A->cols) * static_cast<size_t>(n);
  OFSPMM_CUDA_OK(cudaMemsetAsync(acc, 0, out_elems * sizeof(float), stream));
  BwdAtomicParams p;
  p.crow = A->crow;
  p.col = A->col;
  p.val = A->val;
  p.dY = dY;
  p.acc = acc;
  p.part = part;
  p.cols = A->cols;
  p.rows = static_cast<int>(A->rows);
  p.n = static_cast<int>(n);
  p.P = static_cast<int>(P);
  const bool aligned = ((reinterpret_cast<uintptr_t>(dY) | reinterpret_cast<uintptr_t>(acc)) & 15) == 0;
  const LaneLayout l = lane_layout(LaneOp::kAtomic, dense_dtype, n, aligned);
  const int rc = dispatch_index<true>(A->idx_dtype, wide_nnz(A->nnz), [&](auto idx, auto part) {
    return dispatch_dtypes<true>(dense_dtype, A->val_dtype, [&](auto dense, auto val) {
      return launch_typed<typename decltype(dense)::type, typename decltype(val)::type, typename decltype(idx)::type,
                          typename decltype(part)::type>(p, l, stream);
    });
  });
  if (rc != OFSPMM_OK || dB_cast_out == nullptr) return rc;
  // bf16 output: cast the fp32 accumulator once
  DevInfo dev;
  if (int rc2 = get_dev_info(&dev)) return rc2;
  cast_from_f32_kernel<__nv_bfloat16><<<dev.sms * 8, 256, 0, stream>>>(
      acc, static_cast<__nv_bfloat16*>(dB_cast_out), static_cast<long long>(out_elems));
  return launched();
}

}  // namespace ofspmm
