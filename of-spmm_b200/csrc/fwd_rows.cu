// fwd_rows.cu — the whole-row family (spmm_rows_kernel.cuh): one launch, no workspace; picked by
// ofspmm_choose_variant for small problems whose longest row is short.
#include "internal.h"
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

template <typename DT, typename ValT>
int launch_rows_typed(const FwdParams& p, cudaStream_t stream) {
  constexpr int VECW = 16 / sizeof(DT);
  const int nvec = p.n / VECW;
  if (nvec <= 8) return launch_rows_one<DT, ValT, VECW, 8>(p, stream);
  if (nvec <= 16) return launch_rows_one<DT, ValT, VECW, 16>(p, stream);
  return launch_rows_one<DT, ValT, VECW, 32>(p, stream);
}

}  // namespace

// Preconditions (checked by the caller, fwd.cu:rows_kernel_applies): int32 indices, 16-byte
// aligned rows, n a multiple of the 16-byte vector and at most 32 vectors wide.
int launch_family_rows(const FwdParams& p, int dense_dtype, int val_dtype, cudaStream_t stream) {
  if (dense_dtype == OFSPMM_DTYPE_FLOAT && val_dtype == OFSPMM_DTYPE_FLOAT) return launch_rows_typed<float, float>(p, stream);
  if (dense_dtype == OFSPMM_DTYPE_BFLOAT16 && val_dtype == OFSPMM_DTYPE_FLOAT) return launch_rows_typed<__nv_bfloat16, float>(p, stream);
  if (dense_dtype == OFSPMM_DTYPE_BFLOAT16 && val_dtype == OFSPMM_DTYPE_BFLOAT16)
    return launch_rows_typed<__nv_bfloat16, __nv_bfloat16>(p, stream);
  if (dense_dtype == OFSPMM_DTYPE_FLOAT && val_dtype == OFSPMM_VAL_UNIT) return launch_rows_typed<float, UnitVal>(p, stream);
  if (dense_dtype == OFSPMM_DTYPE_BFLOAT16 && val_dtype == OFSPMM_VAL_UNIT) return launch_rows_typed<__nv_bfloat16, UnitVal>(p, stream);
  return OFSPMM_ERR_UNSUPPORTED_DTYPE;
}

}  // namespace ofspmm
