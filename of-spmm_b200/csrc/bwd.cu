// bwd.cu — launch of the atomic A^T·dY scatter (route 2 of ofspmm_bwd_b).
#include "internal.h"
#include "sddmm_bwd_kernels.cuh"

namespace ofspmm {

namespace {

template <typename DT, typename ValT, typename IdxT, typename PartT, int VEC, int LPR, int CH>
int launch_one(const BwdAtomicParams& p, int panels, cudaStream_t stream) {
  constexpr int ITEMS = kTaskItems;
  constexpr int WARPS = kWarpsPerCta;
  auto kern = bwd_atomic_kernel<DT, ValT, IdxT, VEC, LPR, CH, ITEMS, WARPS, PartT>;
  const size_t smem = sizeof(TaskStage<IdxT, ValT, ITEMS>) * WARPS + sizeof(uint64_t) * WARPS;
  OFSPMM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  int occ = 0;
  OFSPMM_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, WARPS * 32, smem));
  if (occ < 1) return OFSPMM_ERR_CUDA;
  const int64_t ctas_needed = (static_cast<int64_t>(p.P) + WARPS - 1) / WARPS;
  int64_t per_panel = static_cast<int64_t>(dev.sms) * occ / panels;
  if (per_panel < dev.sms) per_panel = dev.sms;
  const int gx = static_cast<int>(ctas_needed < per_panel ? ctas_needed : per_panel);
  kern<<<dim3(gx, panels), WARPS * 32, smem, stream>>>(p);
  count_launch();
  OFSPMM_CUDA_OK(cudaGetLastError());
  return OFSPMM_OK;
}

template <typename DT, typename ValT, typename IdxT, typename PartT>
int launch_typed(const BwdAtomicParams& p, bool aligned, cudaStream_t stream) {
  constexpr int VECW = 16 / sizeof(DT);
  const int n = p.n;
  if (aligned && n % VECW == 0) {
    const int nvec = n / VECW;
    if (nvec <= 8) return launch_one<DT, ValT, IdxT, PartT, VECW, 8, 1>(p, 1, stream);
    if (nvec <= 16) return launch_one<DT, ValT, IdxT, PartT, VECW, 16, 1>(p, 1, stream);
    if (nvec <= 32) return launch_one<DT, ValT, IdxT, PartT, VECW, 32, 1>(p, 1, stream);
    if (nvec <= 64) return launch_one<DT, ValT, IdxT, PartT, VECW, 32, 2>(p, 1, stream);
    return launch_one<DT, ValT, IdxT, PartT, VECW, 32, 4>(p, (nvec + 127) / 128, stream);
  }
  if (n <= 32) return launch_one<DT, ValT, IdxT, PartT, 1, 32, 1>(p, 1, stream);
  if (n <= 128) return launch_one<DT, ValT, IdxT, PartT, 1, 32, 4>(p, 1, stream);
  return launch_one<DT, ValT, IdxT, PartT, 1, 32, 8>(p, (n + 255) / 256, stream);
}

template <typename IdxT, typename PartT>
int launch_idx(const BwdAtomicParams& p, int dense_dtype, int val_dtype, bool aligned, cudaStream_t stream) {
  if (dense_dtype == OFSPMM_DTYPE_FLOAT && val_dtype == OFSPMM_DTYPE_FLOAT)
    return launch_typed<float, float, IdxT, PartT>(p, aligned, stream);
  if (dense_dtype == OFSPMM_DTYPE_BFLOAT16 && val_dtype == OFSPMM_DTYPE_FLOAT)
    return launch_typed<__nv_bfloat16, float, IdxT, PartT>(p, aligned, stream);
  if (dense_dtype == OFSPMM_DTYPE_BFLOAT16 && val_dtype == OFSPMM_DTYPE_BFLOAT16)
    return launch_typed<__nv_bfloat16, __nv_bfloat16, IdxT, PartT>(p, aligned, stream);
  if (dense_dtype == OFSPMM_DTYPE_FLOAT && val_dtype == OFSPMM_VAL_UNIT)
    return launch_typed<float, UnitVal, IdxT, PartT>(p, aligned, stream);
  if (dense_dtype == OFSPMM_DTYPE_BFLOAT16 && val_dtype == OFSPMM_VAL_UNIT)
    return launch_typed<__nv_bfloat16, UnitVal, IdxT, PartT>(p, aligned, stream);
  return OFSPMM_ERR_UNSUPPORTED_DTYPE;
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
  int rc = OFSPMM_ERR_UNSUPPORTED_DTYPE;
  if (A->idx_dtype == OFSPMM_DTYPE_INT32) rc = launch_idx<int32_t, int2>(p, dense_dtype, A->val_dtype, aligned, stream);
  if (A->idx_dtype == OFSPMM_DTYPE_INT64 && !wide_nnz(A->nnz))
    rc = launch_idx<int64_t, int2>(p, dense_dtype, A->val_dtype, aligned, stream);
  if (A->idx_dtype == OFSPMM_DTYPE_INT64 && wide_nnz(A->nnz))
    rc = launch_idx<int64_t, longlong2>(p, dense_dtype, A->val_dtype, aligned, stream);
  if (rc != OFSPMM_OK) return rc;
  if (dB_cast_out != nullptr) {  // bf16 output: cast the fp32 accumulator once
    DevInfo dev;
    if (int rc2 = get_dev_info(&dev)) return rc2;
    cast_from_f32_kernel<__nv_bfloat16><<<dev.sms * 8, 256, 0, stream>>>(
        acc, static_cast<__nv_bfloat16*>(dB_cast_out), static_cast<long long>(out_elems));
    count_launch();
    OFSPMM_CUDA_OK(cudaGetLastError());
  }
  return OFSPMM_OK;
}

}  // namespace ofspmm
