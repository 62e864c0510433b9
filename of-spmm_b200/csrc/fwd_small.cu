// fwd_small.cu — small-problem forward family: 64 merge items per task, so a matrix that would
// not fill the GPU with 256-item tasks spreads over 4x more warps (latency-bound regime).
#include "fwd_launch.cuh"

namespace ofspmm {
int launch_family_small(const FwdParams& p, const LaneLayout& l, int idx_dtype, int dense_dtype, int val_dtype,
                        const FwdLaunch& L, cudaStream_t stream) {
  return launch_family<false, kSmallTaskItems>(p, l, idx_dtype, dense_dtype, val_dtype, L, stream);
}
}  // namespace ofspmm
