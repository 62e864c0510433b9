// fwd_base.cu — the default forward family: 256 merge items per task, nnz-parallel lanes.
#include "fwd_launch.cuh"

namespace ofspmm {
int launch_family_base(const FwdParams& p, const LaneLayout& l, int idx_dtype, int dense_dtype, int val_dtype,
                       const FwdLaunch& L, cudaStream_t stream) {
  return launch_family<false, kTaskItems>(p, l, idx_dtype, dense_dtype, val_dtype, L, stream);
}
}  // namespace ofspmm
