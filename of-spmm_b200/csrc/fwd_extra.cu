// fwd_extra.cu — histogram-selected forward family: the row-parallel layout (each group of 8 / 16
// lanes owns whole rows, 4 / 2 rows in flight per warp) for graphs whose typical row is shorter
// than the 16 non-zeros one warp instruction of the nnz-parallel layout consumes.
#include "fwd_launch.cuh"

namespace ofspmm {
int launch_family_rowpar(const FwdParams& p, const LaneLayout& l, int idx_dtype, int dense_dtype, int val_dtype,
                         const FwdLaunch& L, cudaStream_t stream) {
  return launch_family<true, kTaskItems>(p, l, idx_dtype, dense_dtype, val_dtype, L, stream);
}
}  // namespace ofspmm
