// build.cu — graph construction on the device (SURVEY.md §8f rank 1): the step BEFORE the SpMM path.
//   * COO edge list -> CSR: stable radix sort of the (row, col) keys (cub::DeviceRadixSort, the
//     library primitive the transpose already uses), then hand-written kernels that flag segment
//     heads, coalesce duplicates in source order (sum / max / first — deterministic), emit the
//     column / value arrays and binary-search the row offsets.  Entries outside the matrix are
//     dropped and counted.
//   * row expansion (CSR -> COO rows), |A| row sums, symmetric / row normalisation (the GCN
//     propagation matrix D^-1/2 A D^-1/2 of configs[4]).
// One-off, off the per-step path; the reference has only unique / arg-sort style primitives to
// build such a pipeline from (oneflow/core/cuda/unique.cuh, oneflow/user/kernels/arg_sort_kernel.cu).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "launch.cuh"

namespace ofspmm {

namespace {

__global__ void coo_keys_kernel(const long long* __restrict__ row, const long long* __restrict__ col, long long n,
                                long long rows, long long cols, long long* __restrict__ keys, long long* __restrict__ idx) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  const long long sentinel = rows * cols;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const long long r = row[i], c = col[i];
    const bool ok = r >= 0 && r < rows && c >= 0 && c < cols;
    keys[i] = ok ? r * cols + c : sentinel;   // dropped entries sort behind every valid key
    idx[i] = i;
  }
}

__global__ void coo_heads_kernel(const long long* __restrict__ keys, long long n, long long sentinel,
                                 int* __restrict__ flag) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
    flag[i] = keys[i] < sentinel && (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
}

// One thread per segment head: walks its run of equal keys in sorted (= source, the sort is stable)
// order, so "sum" adds in a fixed order and "first" is the first occurrence in the edge list.
template <typename IdxT>
__global__ void coo_coalesce_kernel(const long long* __restrict__ keys, const long long* __restrict__ perm,
                                    const int* __restrict__ flag, const int* __restrict__ pos,
                                    const float* __restrict__ val, long long n, long long cols, int mode,
                                    IdxT* __restrict__ col_out, float* __restrict__ val_out,
                                    long long* __restrict__ ukeys) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    if (!flag[i]) continue;
    const long long key = keys[i];
    float acc = val != nullptr ? val[perm[i]] : 1.0f;
    if (mode != 2) {
      for (long long j = i + 1; j < n && keys[j] == key; ++j) {
        const float v = val != nullptr ? val[perm[j]] : 1.0f;
        acc = mode == 0 ? acc + v : fmaxf(acc, v);
      }
    }
    const int p = pos[i];
    col_out[p] = static_cast<IdxT>(key % cols);
    val_out[p] = acc;
    ukeys[p] = key;
  }
}

// crow[r] = number of unique entries with row < r; also reports the counts.
template <typename IdxT>
__global__ void coo_offsets_kernel(const long long* __restrict__ ukeys, const long long* __restrict__ sorted_keys,
                                   const int* __restrict__ flag, const int* __restrict__ pos, long long n,
                                   long long rows, long long cols, IdxT* __restrict__ crow,
                                   long long* __restrict__ counts) {
  const long long r = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long unique = n > 0 ? static_cast<long long>(pos[n - 1]) + flag[n - 1] : 0;
  if (r == 0 && counts != nullptr) {
    counts[0] = unique;
    // dropped = entries whose key is the sentinel: they are the tail of the sorted keys
    long long lo = 0, hi = n;
    const long long sentinel = rows * cols;
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if (sorted_keys[mid] < sentinel) lo = mid + 1; else hi = mid;
    }
    counts[1] = n - lo;
  }
  if (r > rows) return;
  const long long target = r * cols;
  long long lo = 0, hi = unique;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (ukeys[mid] < target) lo = mid + 1; else hi = mid;
  }
  crow[r] = static_cast<IdxT>(lo);
}

template <typename IdxT>
__global__ void expand_rows_kernel(const IdxT* __restrict__ crow, long long rows, long long* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  for (long long r = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps) {
    const long long b = static_cast<long long>(crow[r]), e = static_cast<long long>(crow[r + 1]);
    for (long long p = b + lane; p < e; p += 32) out[p] = r;
  }
}

// dinv[r] = f(sum_p |val[p]|) over row r: mode 0 -> rsqrt (symmetric), 1 -> reciprocal (row mean); 0 for empty rows
template <typename IdxT>
__global__ void row_dinv_kernel(const IdxT* __restrict__ crow, const float* __restrict__ val, long long rows, int mode,
                                float* __restrict__ dinv) {
  const int lane = threadIdx.x & 31;
  const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  for (long long r = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps) {
    const long long b = static_cast<long long>(crow[r]), e = static_cast<long long>(crow[r + 1]);
    float s = 0.f;
    for (long long p = b + lane; p < e; p += 32) s += fabsf(val[p]);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if (lane == 0) dinv[r] = s > 0.f ? (mode == 0 ? rsqrtf(s) : 1.0f / s) : 0.f;
  }
}

template <typename IdxT>
__global__ void scale_kernel(const IdxT* __restrict__ crow, const IdxT* __restrict__ col, long long rows,
                             long long cols, int mode, const float* __restrict__ dinv, float* __restrict__ val) {
  const int lane = threadIdx.x & 31;
  const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  for (long long r = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps) {
    const long long b = static_cast<long long>(crow[r]), e = static_cast<long long>(crow[r + 1]);
    const float dr = dinv[r];
    for (long long p = b + lane; p < e; p += 32) {
      float s = dr;
      if (mode == 0) {
        const long long c = static_cast<long long>(col[p]);
        s *= (c >= 0 && c < cols) ? dinv[c] : 0.f;
      }
      val[p] *= s;
    }
  }
}

int key_bits(int64_t rows, int64_t cols) {
  const unsigned long long maxkey = static_cast<unsigned long long>(rows) * static_cast<unsigned long long>(cols);
  int b = 1;
  while (b < 63 && (1ull << b) <= maxkey) ++b;
  return b;
}

struct CooLayout {
  size_t keys_in, keys_out, idx_in, perm, flag, pos, ukeys, cub_tmp, cub_bytes, total;
};

CooLayout coo_layout(int64_t n, int64_t rows, int64_t cols) {
  CooLayout L;
  const size_t a64 = static_cast<size_t>(n > 0 ? n : 1) * sizeof(long long);
  const size_t a32 = static_cast<size_t>(n > 0 ? n : 1) * sizeof(int);
  Carve c;
  L.keys_in = c.take(a64);
  L.keys_out = c.take(a64);
  L.idx_in = c.take(a64);
  L.perm = c.take(a64);
  L.ukeys = c.take(a64);
  L.flag = c.take(a32);
  L.pos = c.take(a32);
  size_t sort_bytes = 0, scan_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, static_cast<const long long*>(nullptr), static_cast<long long*>(nullptr),
                                  static_cast<const long long*>(nullptr), static_cast<long long*>(nullptr),
                                  static_cast<long long>(n), 0, key_bits(rows, cols));
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, static_cast<const int*>(nullptr), static_cast<int*>(nullptr),
                                static_cast<long long>(n));
  L.cub_bytes = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
  L.cub_tmp = c.take(L.cub_bytes);
  L.total = c.total;
  return L;
}

template <typename IdxT>
int coo_impl(const int64_t* row, const int64_t* col, const float* val, int64_t n, int64_t rows, int64_t cols, int mode,
             void* crow, void* col_out, float* val_out, int64_t* counts, void* ws, cudaStream_t stream) {
  const CooLayout L = coo_layout(n, rows, cols);
  unsigned char* w = static_cast<unsigned char*>(ws);
  long long* keys_in = reinterpret_cast<long long*>(w + L.keys_in);
  long long* keys_out = reinterpret_cast<long long*>(w + L.keys_out);
  long long* idx_in = reinterpret_cast<long long*>(w + L.idx_in);
  long long* perm = reinterpret_cast<long long*>(w + L.perm);
  long long* ukeys = reinterpret_cast<long long*>(w + L.ukeys);
  int* flag = reinterpret_cast<int*>(w + L.flag);
  int* pos = reinterpret_cast<int*>(w + L.pos);
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  const int grid = dev.sms * 8;
  if (n > 0) {
    coo_keys_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const long long*>(row), reinterpret_cast<const long long*>(col),
                                              n, rows, cols, keys_in, idx_in);
    count_launch();
    size_t cub_bytes = L.cub_bytes;
    OFSPMM_CUDA_OK(cub::DeviceRadixSort::SortPairs(w + L.cub_tmp, cub_bytes, static_cast<const long long*>(keys_in), keys_out,
                                                   static_cast<const long long*>(idx_in), perm, static_cast<long long>(n), 0,
                                                   key_bits(rows, cols), stream));
    coo_heads_kernel<<<grid, 256, 0, stream>>>(keys_out, n, rows * cols, flag);
    count_launch();
    cub_bytes = L.cub_bytes;
    OFSPMM_CUDA_OK(cub::DeviceScan::ExclusiveSum(w + L.cub_tmp, cub_bytes, static_cast<const int*>(flag), pos,
                                                 static_cast<long long>(n), stream));
    count_launch(6);
    coo_coalesce_kernel<IdxT><<<grid, 256, 0, stream>>>(keys_out, perm, flag, pos, val, n, cols, mode,
                                                        static_cast<IdxT*>(col_out), val_out, ukeys);
    count_launch();
  }
  coo_offsets_kernel<IdxT><<<static_cast<unsigned>((rows + 1 + 255) / 256), 256, 0, stream>>>(
      ukeys, keys_out, flag, pos, n, rows, cols, static_cast<IdxT*>(crow), reinterpret_cast<long long*>(counts));
  return launched();
}

}  // namespace

size_t coo_to_csr_workspace_bytes(int64_t n, int64_t rows, int64_t cols) { return coo_layout(n, rows, cols).total; }

int launch_coo_to_csr(const int64_t* row, const int64_t* col, const float* val, int64_t n, int64_t rows, int64_t cols,
                      int mode, int idx_dtype, void* crow, void* col_out, float* val_out, int64_t* counts, void* ws,
                      size_t ws_bytes, cudaStream_t stream) {
  if (ws == nullptr || ws_bytes < coo_layout(n, rows, cols).total) return OFSPMM_ERR_WORKSPACE;
  return dispatch_idx(idx_dtype, [&](auto idx) {
    return coo_impl<typename decltype(idx)::type>(row, col, val, n, rows, cols, mode, crow, col_out, val_out, counts, ws,
                                                  stream);
  });
}

int launch_expand_rows(const void* crow, int idx_dtype, int64_t rows, int64_t* out, cudaStream_t stream) {
  if (rows == 0) return OFSPMM_OK;
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  const int grid = dev.sms * 8;
  return dispatch_idx(idx_dtype, [&](auto idx) {
    using IdxT = typename decltype(idx)::type;
    expand_rows_kernel<IdxT><<<grid, 256, 0, stream>>>(static_cast<const IdxT*>(crow), rows, reinterpret_cast<long long*>(out));
    return launched();
  });
}

int launch_csr_normalize(const void* crow, const void* col, float* val, int idx_dtype, int64_t rows, int64_t cols, int mode,
                         float* dinv, cudaStream_t stream) {
  if (rows == 0) return OFSPMM_OK;
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  const int grid = dev.sms * 8;
  return dispatch_idx(idx_dtype, [&](auto idx) {
    using IdxT = typename decltype(idx)::type;
    row_dinv_kernel<IdxT><<<grid, 256, 0, stream>>>(static_cast<const IdxT*>(crow), val, rows, mode, dinv);
    scale_kernel<IdxT><<<grid, 256, 0, stream>>>(static_cast<const IdxT*>(crow), static_cast<const IdxT*>(col), rows, cols,
                                                 mode, dinv, val);
    return launched(2);
  });
}

}  // namespace ofspmm
