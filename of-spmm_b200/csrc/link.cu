// link.cu — the device pieces of link prediction (include/ofspmm.h): edge lookup, (u, v) -> the
// position of that entry in A, and negative sampling with rejection of the edges of A and of
// self-loops.  Both are one thread per query or slot with a binary search of one row (the columns
// of a row ascend), no workspace and a fixed-size output.
#include "bsearch.cuh"
#include "launch.cuh"
#include "sample_key.h"

namespace ofspmm {

namespace {

// Position of the first entry of row u equal to c, or -1 (also for u outside [0, rows)).
template <typename IdxT>
__device__ __forceinline__ long long find_entry(const IdxT* __restrict__ crow, const IdxT* __restrict__ col,
                                                long long rows, long long u, IdxT c) {
  if (u < 0 || u >= rows) return -1;
  const long long b = static_cast<long long>(crow[u]), e = static_cast<long long>(crow[u + 1]);
  const long long p = b + lower_bound(col + b, e - b, c);
  return p < e && col[p] == c ? p : -1;
}

template <typename IdxT>
__global__ void edge_ids_kernel(const IdxT* __restrict__ crow, const IdxT* __restrict__ col, long long rows,
                                const IdxT* __restrict__ u, const IdxT* __restrict__ v, long long n,
                                IdxT* __restrict__ eid) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
    eid[i] = static_cast<IdxT>(find_entry(crow, col, rows, static_cast<long long>(u[i]), v[i]));
}

// One thread per slot (i, t) of the (num_src x k) output (one per source when k == 0, so that
// invalid sources are still counted); counts[0] += slots left at -1, counts[1] += invalid sources.
template <typename IdxT>
__global__ void negative_sample_kernel(const IdxT* __restrict__ crow, const IdxT* __restrict__ col, long long rows,
                                       long long cols, const IdxT* __restrict__ src, long long num_src, long long k,
                                       unsigned long long seed, unsigned flags, int max_trials,
                                       IdxT* __restrict__ neg, unsigned long long* __restrict__ counts) {
  const long long per = k > 0 ? k : 1;
  const long long n = num_src * per;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  unsigned long long failed = 0, invalid = 0;
  for (long long s = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; s < n; s += stride) {
    const long long i = s / per, t = s - i * per;
    const long long u = static_cast<long long>(src[i]);
    const bool valid = u >= 0 && u < rows;
    if (!valid && t == 0) ++invalid;
    if (k == 0) continue;
    long long c = -1;
    if (valid && cols > 0) {
      const unsigned long long h0 = sk_mix64(seed ^ static_cast<unsigned long long>(i));
      for (int r = 0; r < max_trials; ++r) {
        const unsigned long long x =
            sk_mix64(h0 + static_cast<unsigned long long>(r) * static_cast<unsigned long long>(k) +
                     static_cast<unsigned long long>(t));
        const long long p = static_cast<long long>(__umul64hi(x, static_cast<unsigned long long>(cols)));
        if ((flags & OFSPMM_NEG_EXCLUDE_SELF) && p == u) continue;
        if ((flags & OFSPMM_NEG_EXCLUDE_EDGES) && find_entry(crow, col, rows, u, static_cast<IdxT>(p)) >= 0) continue;
        c = p;
        break;
      }
    }
    if (c < 0) ++failed;
    neg[s] = static_cast<IdxT>(c);
  }
  failed = __reduce_add_sync(0xffffffffu, static_cast<unsigned>(failed));
  invalid = __reduce_add_sync(0xffffffffu, static_cast<unsigned>(invalid));
  if ((threadIdx.x & 31) == 0) {
    if (failed) atomicAdd(&counts[0], failed);
    if (invalid) atomicAdd(&counts[1], invalid);
  }
}

}  // namespace

int launch_edge_ids(const ofspmm_csr* A, const void* u, const void* v, int64_t n, void* eid, cudaStream_t stream) {
  if (n == 0) return OFSPMM_OK;
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  return dispatch_idx(A->idx_dtype, [&](auto idx) {
    using IdxT = typename decltype(idx)::type;
    edge_ids_kernel<IdxT><<<grid_for(n, 256, dev.sms * 8, dev.sms), 256, 0, stream>>>(
        static_cast<const IdxT*>(A->crow), static_cast<const IdxT*>(A->col), A->rows, static_cast<const IdxT*>(u),
        static_cast<const IdxT*>(v), n, static_cast<IdxT*>(eid));
    return launched();
  });
}

int launch_negative_sample(const ofspmm_csr* A, const void* src, int64_t num_src, int64_t k, uint64_t seed,
                           uint32_t flags, int max_trials, void* neg_dst, int64_t* counts, cudaStream_t stream) {
  OFSPMM_CUDA_OK(cudaMemsetAsync(counts, 0, 2 * sizeof(int64_t), stream));
  if (num_src == 0) return OFSPMM_OK;
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  const long long slots = num_src * (k > 0 ? k : 1);
  return dispatch_idx(A->idx_dtype, [&](auto idx) {
    using IdxT = typename decltype(idx)::type;
    negative_sample_kernel<IdxT><<<grid_for(slots, 256, dev.sms * 8, dev.sms), 256, 0, stream>>>(
        static_cast<const IdxT*>(A->crow), static_cast<const IdxT*>(A->col), A->rows, A->cols,
        static_cast<const IdxT*>(src), num_src, k, seed, flags, max_trials, static_cast<IdxT*>(neg_dst),
        reinterpret_cast<unsigned long long*>(counts));
    return launched();
  });
}

}  // namespace ofspmm
