// fwd_rows.cu — the whole-row family (spmm_rows_kernel.cuh): one launch, no workspace; picked by
// ofspmm_choose_variant for small problems whose longest row is short.
#include "launch.cuh"
#include "spmm_rows_kernel.cuh"

namespace ofspmm {

namespace {

template <typename DT, typename ValT, int VEC, int LPR>
int launch_rows_one(const FwdParams& p, cudaStream_t stream) {
  constexpr int rows_per_cta = kRowsKernelWarps * (32 / LPR);
  const unsigned grid = static_cast<unsigned>((static_cast<int64_t>(p.rows) + rows_per_cta - 1) / rows_per_cta);
  spmm_rows_kernel<DT, ValT, VEC, LPR><<<grid, kRowsKernelWarps * 32, 0, stream>>>(p);
  count_launch();
  OFSPMM_CUDA_OK(cudaGetLastError());
  return OFSPMM_OK;
}

}  // namespace

// Preconditions (checked by the caller, fwd.cu:rows_layout): int32 indices, 16-byte aligned rows
// and a layout of the whole-row ladder.
int launch_family_rows(const FwdParams& p, const LaneLayout& l, int dense_dtype, int val_dtype, cudaStream_t stream) {
  return dispatch_dtypes<true>(dense_dtype, val_dtype, [&](auto dense, auto val) {
    using DT = typename decltype(dense)::type;
    constexpr int V = vec_width(sizeof(DT));
    return dispatch_lanes<Lanes<V, 8, 1>, Lanes<V, 16, 1>, Lanes<V, 32, 1>>(l, [&](auto lanes) {
      return launch_rows_one<DT, typename decltype(val)::type, decltype(lanes)::VEC, decltype(lanes)::LPR>(p, stream);
    });
  });
}

}  // namespace ofspmm
