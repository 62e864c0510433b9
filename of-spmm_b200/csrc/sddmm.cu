// sddmm.cu — variant selection and launch of the SDDMM value-gradient kernels.
#include "internal.h"
#include "sddmm_bwd_kernels.cuh"

namespace ofspmm {

namespace {

template <typename Kern>
int launch_persistent(Kern kern, SddmmParams p, size_t smem, bool dynamic_ok, KernelLaunchCache& cache, cudaStream_t stream) {
  constexpr int WARPS = kWarpsPerCta;
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  int occ = cache.get(dev.ordinal);  // per (kernel, device) launch constants, queried once
  if (occ == 0) {
    OFSPMM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    OFSPMM_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, WARPS * 32, smem));
    if (occ < 1) return OFSPMM_ERR_CUDA;
    cache.set(dev.ordinal, occ);
  }
  const int64_t ctas_needed = (static_cast<int64_t>(p.P) + WARPS - 1) / WARPS;
  const int64_t resident = static_cast<int64_t>(dev.sms) * occ;
  const int gx = static_cast<int>(ctas_needed < resident ? ctas_needed : resident);
  if (!dynamic_ok || gx == ctas_needed) p.counter = nullptr;
  if (p.counter != nullptr) OFSPMM_CUDA_OK(cudaMemsetAsync(p.counter, 0, sizeof(unsigned int), stream));
  kern<<<gx, WARPS * 32, smem, stream>>>(p);
  count_launch();
  OFSPMM_CUDA_OK(cudaGetLastError());
  return OFSPMM_OK;
}

template <typename DT, typename ValT, typename IdxT, typename PartT, int VEC, int LPR, int CH>
int launch_one(const SddmmParams& p, cudaStream_t stream) {
  constexpr int ITEMS = kTaskItems;
  constexpr int WARPS = kWarpsPerCta;
  const size_t smem = sizeof(TaskStage<IdxT, float, ITEMS>) * WARPS + sizeof(uint64_t) * WARPS;
  static KernelLaunchCache cache_full, cache_masked;
  if (p.n % (LPR * VEC * CH) == 0)
    return launch_persistent(sddmm_merge_kernel<DT, ValT, IdxT, VEC, LPR, CH, true, ITEMS, WARPS, PartT>, p, smem, true, cache_full, stream);
  return launch_persistent(sddmm_merge_kernel<DT, ValT, IdxT, VEC, LPR, CH, false, ITEMS, WARPS, PartT>, p, smem, true, cache_masked, stream);
}

template <typename DT, typename ValT, typename IdxT, typename PartT, int VEC>
int launch_wide(const SddmmParams& p, cudaStream_t stream) {
  constexpr int ITEMS = kTaskItems;
  constexpr int WARPS = kWarpsPerCta;
  const size_t smem = sizeof(TaskStage<IdxT, float, ITEMS>) * WARPS + sizeof(uint64_t) * WARPS;
  static KernelLaunchCache cache;
  return launch_persistent(sddmm_wide_kernel<DT, ValT, IdxT, VEC, ITEMS, WARPS, PartT>, p, smem, false, cache, stream);
}

template <typename DT, typename ValT, typename IdxT, typename PartT>
int launch_typed(const SddmmParams& p, bool aligned, cudaStream_t stream) {
  constexpr int VECW = 16 / sizeof(DT);
  const int n = p.n;
  if (aligned && n % VECW == 0) {
    const int nvec = n / VECW;
    if (nvec <= 8) return launch_one<DT, ValT, IdxT, PartT, VECW, 8, 1>(p, stream);
    if (nvec <= 16) return launch_one<DT, ValT, IdxT, PartT, VECW, 16, 1>(p, stream);
    if (nvec <= 32) return launch_one<DT, ValT, IdxT, PartT, VECW, 32, 1>(p, stream);
    if (nvec <= 64) return launch_one<DT, ValT, IdxT, PartT, VECW, 32, 2>(p, stream);
    if (nvec <= 128) return launch_one<DT, ValT, IdxT, PartT, VECW, 32, 4>(p, stream);
    return launch_wide<DT, ValT, IdxT, PartT, VECW>(p, stream);
  }
  if (n <= 32) return launch_one<DT, ValT, IdxT, PartT, 1, 32, 1>(p, stream);
  if (n <= 128) return launch_one<DT, ValT, IdxT, PartT, 1, 32, 4>(p, stream);
  return launch_wide<DT, ValT, IdxT, PartT, 1>(p, stream);
}

template <typename IdxT, typename PartT>
int launch_idx(const SddmmParams& p, int dense_dtype, int val_dtype, bool aligned, cudaStream_t stream) {
  if (dense_dtype == OFSPMM_DTYPE_FLOAT && val_dtype == OFSPMM_DTYPE_FLOAT)
    return launch_typed<float, float, IdxT, PartT>(p, aligned, stream);
  if (dense_dtype == OFSPMM_DTYPE_BFLOAT16 && val_dtype == OFSPMM_DTYPE_FLOAT)
    return launch_typed<__nv_bfloat16, float, IdxT, PartT>(p, aligned, stream);
  if (dense_dtype == OFSPMM_DTYPE_BFLOAT16 && val_dtype == OFSPMM_DTYPE_BFLOAT16)
    return launch_typed<__nv_bfloat16, __nv_bfloat16, IdxT, PartT>(p, aligned, stream);
  return OFSPMM_ERR_UNSUPPORTED_DTYPE;
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
  if (A->idx_dtype == OFSPMM_DTYPE_INT32) return launch_idx<int32_t, int2>(p, dense_dtype, A->val_dtype, aligned, stream);
  if (A->idx_dtype == OFSPMM_DTYPE_INT64 && !wide_nnz(A->nnz))
    return launch_idx<int64_t, int2>(p, dense_dtype, A->val_dtype, aligned, stream);
  if (A->idx_dtype == OFSPMM_DTYPE_INT64) return launch_idx<int64_t, longlong2>(p, dense_dtype, A->val_dtype, aligned, stream);
  return OFSPMM_ERR_UNSUPPORTED_DTYPE;
}

}  // namespace ofspmm
