// misc.cu — public merge-path partitioner, row-length histogram and the one-off device
// CSR -> CSR(A^T) transpose (plan / OpKernelState construction; not on the per-step path).
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"
#include "internal.h"

namespace ofspmm {

namespace {

template <typename IdxT>
__global__ void partition_public_kernel(const IdxT* __restrict__ crow, long long rows, long long nnz,
                                        long long parts, long long* __restrict__ out_row,
                                        long long* __restrict__ out_nz) {
  const long long k = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k > parts) return;
  const long long total = rows + nnz;
  const long long ipw = parts > 0 ? (total + parts - 1) / parts : total;
  long long d = k * ipw;
  if (d > total) d = total;
  const long long r = merge_path_search<IdxT>(crow, rows, nnz, d);
  out_row[k] = r;
  out_nz[k] = d - r;
}

template <typename IdxT>
__global__ void row_hist_kernel(const IdxT* __restrict__ crow, long long rows,
                                unsigned long long* __restrict__ hist) {
  __shared__ unsigned int sh[32];
  if (threadIdx.x < 32) sh[threadIdx.x] = 0;
  __syncthreads();
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < rows; i += stride) {
    const long long len = static_cast<long long>(crow[i + 1]) - static_cast<long long>(crow[i]);
    int b = len <= 0 ? 0 : 64 - __clzll(len);
    if (b > 31) b = 31;
    atomicAdd(&sh[b], 1u);
  }
  __syncthreads();
  if (threadIdx.x < 32 && sh[threadIdx.x] != 0)
    atomicAdd(&hist[threadIdx.x], static_cast<unsigned long long>(sh[threadIdx.x]));
}

// Sort keys of the transpose: the column index, or the sentinel `cols` for an index outside
// [0, cols) — such entries are skipped by every kernel of the library (include/ofspmm.h), so they
// must not alias into a valid column bucket; they sort behind every valid key.  pos[p] = p.
// KeyT is 32-bit whenever the sentinel fits (halves the key buffers of an int64 matrix).
template <typename IdxT, typename KeyT>
__global__ void transpose_keys_kernel(const IdxT* __restrict__ col, long long cols, long long count,
                                      KeyT* __restrict__ keys, IdxT* __restrict__ pos) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += stride) {
    const IdxT c = col[i];
    const bool ok = static_cast<unsigned long long>(c) < static_cast<unsigned long long>(cols);
    keys[i] = ok ? static_cast<KeyT>(c) : static_cast<KeyT>(cols);
    pos[i] = static_cast<IdxT>(i);
  }
}

// t_crow[c] = first position in the column-sorted key array whose key is >= c.  t_crow[cols] is
// pinned to nnz (crow[rows] == nnz is what the merge-path kernels rely on): the skipped entries
// therefore trail the last row of A^T, where the fill kernel marks them with column -1.
template <typename IdxT, typename KeyT>
__global__ void transpose_offsets_kernel(const KeyT* __restrict__ sorted_cols, long long nnz,
                                         long long cols, IdxT* __restrict__ t_crow) {
  const long long c = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c > cols) return;
  if (c == cols) {
    t_crow[c] = static_cast<IdxT>(cols > 0 ? nnz : 0);
    return;
  }
  long long lo = 0, hi = nnz;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (static_cast<long long>(sorted_cols[mid]) < c) lo = mid + 1; else hi = mid;
  }
  t_crow[c] = static_cast<IdxT>(lo);
}

// For transposed position q with source position p = perm[q]: row(p) by binary search in crow.
template <typename IdxT, typename KeyT, typename ValT>
__global__ void transpose_fill_kernel(const IdxT* __restrict__ crow, long long rows,
                                      const ValT* __restrict__ val, const IdxT* __restrict__ perm,
                                      const KeyT* __restrict__ sorted_keys, long long cols,
                                      long long nnz, IdxT* __restrict__ t_col, ValT* __restrict__ t_val) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; q < nnz; q += stride) {
    const long long p = static_cast<long long>(perm[q]);
    if (static_cast<long long>(sorted_keys[q]) >= cols) {  // skipped entry of A: stays skipped in A^T
      t_col[q] = static_cast<IdxT>(-1);
      if (t_val != nullptr) t_val[q] = ValT{};
      continue;
    }
    long long lo = 0, hi = rows;  // largest r with crow[r] <= p
    while (lo < hi) {
      const long long mid = (lo + hi + 1) >> 1;
      if (static_cast<long long>(crow[mid]) <= p) lo = mid; else hi = mid - 1;
    }
    t_col[q] = static_cast<IdxT>(lo);
    if (t_val != nullptr) t_val[q] = val[p];
  }
}

int bits_for(int64_t cols) {
  int b = 1;
  while (b < 63 && (int64_t{1} << b) < cols) ++b;
  return b;
}

template <typename KeyT, typename IdxT>
size_t cub_sort_temp_bytes(int64_t nnz, int end_bit) {
  size_t bytes = 0;
  cub::DoubleBuffer<KeyT> keys(nullptr, nullptr);
  cub::DoubleBuffer<IdxT> vals(nullptr, nullptr);
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, keys, vals, static_cast<long long>(nnz), 0, end_bit);
  return bytes;
}

// Workspace of the transpose: two key buffers and one position buffer for the ping-pong radix
// sort (the other position buffer is t_perm, or t_col when the caller keeps no t_perm: both are
// nnz-long IdxT outputs) and cub's scratch.
struct TransposeLayout {
  size_t keys_a, keys_b, pos, cub_tmp, cub_bytes, total;
};

// Column keys are 32-bit when the sentinel `cols` fits an int32 (every int32 matrix does).
bool narrow_keys(int64_t cols) { return cols < (int64_t{1} << 31) - 1; }

template <typename IdxT, typename KeyT>
TransposeLayout transpose_layout(int64_t cols, int64_t nnz) {
  TransposeLayout L;
  const size_t n = static_cast<size_t>(nnz > 0 ? nnz : 1);
  const size_t karr = align_up(n * sizeof(KeyT), 256);
  L.keys_a = 0;
  L.keys_b = karr;
  L.pos = 2 * karr;
  L.cub_tmp = L.pos + align_up(n * sizeof(IdxT), 256);
  L.cub_bytes = cub_sort_temp_bytes<KeyT, IdxT>(nnz, bits_for(cols + 1));
  L.total = L.cub_tmp + align_up(L.cub_bytes, 256);
  return L;
}

template <typename IdxT, typename KeyT>
int transpose_impl(const ofspmm_csr* A, void* t_crow, void* t_col, void* t_val, void* t_perm,
                   void* ws, size_t ws_bytes, cudaStream_t stream) {
  const int64_t nnz = A->nnz, rows = A->rows, cols = A->cols;
  const TransposeLayout L = transpose_layout<IdxT, KeyT>(cols, nnz);
  if (ws == nullptr || ws_bytes < L.total) return OFSPMM_ERR_WORKSPACE;
  unsigned char* w = static_cast<unsigned char*>(ws);
  cub::DoubleBuffer<KeyT> keys(reinterpret_cast<KeyT*>(w + L.keys_a), reinterpret_cast<KeyT*>(w + L.keys_b));
  IdxT* pos_ws = reinterpret_cast<IdxT*>(w + L.pos);
  cub::DoubleBuffer<IdxT> pos(pos_ws, static_cast<IdxT*>(t_perm != nullptr ? t_perm : t_col));
  // where the sorted positions must end up: t_perm when the caller keeps them, else the workspace
  // buffer; never t_col, which the fill kernel overwrites with rows
  IdxT* perm = t_perm != nullptr ? static_cast<IdxT*>(t_perm) : pos_ws;
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  const int grid = dev.sms * 8;
  if (nnz > 0) {
    transpose_keys_kernel<IdxT, KeyT><<<grid, 256, 0, stream>>>(static_cast<const IdxT*>(A->col), cols, nnz,
                                                                keys.Current(), pos.Current());
    count_launch();
    size_t cub_bytes = L.cub_bytes;
    // stable LSD radix sort by column: entries of one column keep ascending source position,
    // i.e. ascending row — the transposed CSR is deterministic and row-sorted.  The ping-pong
    // overload needs no nnz-long scratch of its own.
    OFSPMM_CUDA_OK(cub::DeviceRadixSort::SortPairs(w + L.cub_tmp, cub_bytes, keys, pos, static_cast<long long>(nnz),
                                                   0, bits_for(cols + 1), stream));
    count_launch(4);
    if (pos.Current() != perm)
      OFSPMM_CUDA_OK(cudaMemcpyAsync(perm, pos.Current(), static_cast<size_t>(nnz) * sizeof(IdxT),
                                     cudaMemcpyDeviceToDevice, stream));
  }
  const KeyT* keys_out = keys.Current();
  IdxT* pos_out = perm;
  transpose_offsets_kernel<IdxT, KeyT><<<static_cast<unsigned>((cols + 1 + 255) / 256), 256, 0, stream>>>(
      keys_out, nnz, cols, static_cast<IdxT*>(t_crow));
  count_launch();
  if (nnz > 0) {
    if (A->val == nullptr || t_val == nullptr) {
      transpose_fill_kernel<IdxT, KeyT, float><<<grid, 256, 0, stream>>>(
          static_cast<const IdxT*>(A->crow), rows, nullptr, pos_out, keys_out, cols, nnz, static_cast<IdxT*>(t_col), nullptr);
    } else if (A->val_dtype == OFSPMM_DTYPE_FLOAT) {
      transpose_fill_kernel<IdxT, KeyT, float><<<grid, 256, 0, stream>>>(
          static_cast<const IdxT*>(A->crow), rows, static_cast<const float*>(A->val), pos_out, keys_out, cols, nnz,
          static_cast<IdxT*>(t_col), static_cast<float*>(t_val));
    } else if (A->val_dtype == OFSPMM_DTYPE_BFLOAT16) {
      transpose_fill_kernel<IdxT, KeyT, __nv_bfloat16><<<grid, 256, 0, stream>>>(
          static_cast<const IdxT*>(A->crow), rows, static_cast<const __nv_bfloat16*>(A->val), pos_out, keys_out, cols, nnz,
          static_cast<IdxT*>(t_col), static_cast<__nv_bfloat16*>(t_val));
    } else {
      return OFSPMM_ERR_UNSUPPORTED_DTYPE;
    }
    count_launch();
  }
  OFSPMM_CUDA_OK(cudaGetLastError());
  return OFSPMM_OK;
}

}  // namespace

int launch_partition_public(const void* crow, int idx_dtype, int64_t rows, int64_t nnz, int64_t parts,
                            int64_t* out_row, int64_t* out_nz, cudaStream_t stream) {
  const unsigned blocks = static_cast<unsigned>((parts + 1 + 255) / 256);
  if (idx_dtype == OFSPMM_DTYPE_INT32) {
    partition_public_kernel<int32_t><<<blocks, 256, 0, stream>>>(
        static_cast<const int32_t*>(crow), rows, nnz, parts, reinterpret_cast<long long*>(out_row),
        reinterpret_cast<long long*>(out_nz));
  } else if (idx_dtype == OFSPMM_DTYPE_INT64) {
    partition_public_kernel<int64_t><<<blocks, 256, 0, stream>>>(
        static_cast<const int64_t*>(crow), rows, nnz, parts, reinterpret_cast<long long*>(out_row),
        reinterpret_cast<long long*>(out_nz));
  } else {
    return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  }
  count_launch();
  OFSPMM_CUDA_OK(cudaGetLastError());
  return OFSPMM_OK;
}

int launch_row_hist(const void* crow, int idx_dtype, int64_t rows, int64_t* hist32, cudaStream_t stream) {
  OFSPMM_CUDA_OK(cudaMemsetAsync(hist32, 0, 32 * sizeof(int64_t), stream));
  if (rows == 0) return OFSPMM_OK;
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  int64_t blocks = (rows + 255) / 256;
  if (blocks > dev.sms * 8) blocks = dev.sms * 8;
  if (idx_dtype == OFSPMM_DTYPE_INT32) {
    row_hist_kernel<int32_t><<<static_cast<unsigned>(blocks), 256, 0, stream>>>(
        static_cast<const int32_t*>(crow), rows, reinterpret_cast<unsigned long long*>(hist32));
  } else if (idx_dtype == OFSPMM_DTYPE_INT64) {
    row_hist_kernel<int64_t><<<static_cast<unsigned>(blocks), 256, 0, stream>>>(
        static_cast<const int64_t*>(crow), rows, reinterpret_cast<unsigned long long*>(hist32));
  } else {
    return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  }
  count_launch();
  OFSPMM_CUDA_OK(cudaGetLastError());
  return OFSPMM_OK;
}

size_t transpose_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz, int idx_dtype) {
  (void)rows;
  if (idx_dtype == OFSPMM_DTYPE_INT32) return transpose_layout<int32_t, int32_t>(cols, nnz).total;
  if (narrow_keys(cols)) return transpose_layout<int64_t, int32_t>(cols, nnz).total;
  return transpose_layout<int64_t, int64_t>(cols, nnz).total;
}

int launch_transpose(const ofspmm_csr* A, void* t_crow, void* t_col, void* t_val, void* t_perm,
                     void* ws, size_t ws_bytes, cudaStream_t stream) {
  if (A->idx_dtype == OFSPMM_DTYPE_INT32) return transpose_impl<int32_t, int32_t>(A, t_crow, t_col, t_val, t_perm, ws, ws_bytes, stream);
  if (A->idx_dtype == OFSPMM_DTYPE_INT64 && narrow_keys(A->cols))
    return transpose_impl<int64_t, int32_t>(A, t_crow, t_col, t_val, t_perm, ws, ws_bytes, stream);
  if (A->idx_dtype == OFSPMM_DTYPE_INT64) return transpose_impl<int64_t, int64_t>(A, t_crow, t_col, t_val, t_perm, ws, ws_bytes, stream);
  return OFSPMM_ERR_UNSUPPORTED_DTYPE;
}

}  // namespace ofspmm
