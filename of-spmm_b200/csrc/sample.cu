// sample.cu — device neighbour sampling (DESIGN.md §3.8): for each destination v, the k = min(deg,
// fanout) entries of row v with the smallest (key, j), key = mix(mix(seed ^ v) + j) (splitmix64), then
// a relabel of the sampled columns into a bipartite block (DGL's block convention: the destinations
// come first in src_nodes, then the other sampled ids in ascending order).
//   count   one thread per destination: validity (range, repeats found in the sorted ids), k, and a
//           list of the rows long enough for a whole CTA;
//   select  one warp per destination (one CTA per long row): radix selection of the k-th smallest
//           key over re-hashed keys, 8 bits per pass, stopping as soon as the bucket holding the
//           k-th key is taken whole; then one pass that emits the selected entries in ascending j
//           (ballot compaction), loading col / val for those only.  A row with deg <= k is copied.
//   relabel radix sort of the sampled ids (cub, as the transpose does), unique / not-a-destination
//           flags, one scan that also compacts away the out-of-range columns, and a binary search
//           per kept entry for its local id.
// Everything the kernels address is sized by (num_dst, cap), never by A's rows.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"
#include "internal.h"

namespace ofspmm {

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kSampleWarps = 8;         // warps per CTA of the warp-per-row kernel
constexpr int kLongThreads = 512;       // threads per CTA of the long-row kernel
constexpr long long kLongRow = 4096;    // rows longer than this are sampled by a whole CTA

__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x *= 0x9E3779B97F4A7C15ull;
  x ^= x >> 30;
  x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27;
  x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return x;
}

// Bits of a sort key that holds ids in [0, rows] (rows itself is the "no id" sentinel).
int id_bits(long long rows) {
  int b = 1;
  while (b < 32 && (1ll << b) <= rows) ++b;
  return b;
}

template <typename T>
__device__ __forceinline__ long long lower_bound(const T* a, long long n, T x) {
  long long lo = 0, hi = n;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (a[mid] < x) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// dkey[i] = dst[i] when it is a row of A, else the sentinel `rows`; didx[i] = i.
template <typename IdxT>
__global__ void sample_dst_keys_kernel(const IdxT* __restrict__ dst, long long num_dst, long long rows,
                                       unsigned* __restrict__ dkey, int* __restrict__ didx) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < num_dst; i += stride) {
    const long long v = static_cast<long long>(dst[i]);
    dkey[i] = static_cast<unsigned>(v >= 0 && v < rows ? v : rows);
    didx[i] = static_cast<int>(i);
  }
}

// kcnt[i] = k of destination i (0 for an invalid one: out of range, or an id that occurs more than
// once); kcnt[num_dst] = 0 so that the exclusive scan ends in the total.
template <typename IdxT>
__global__ void sample_count_kernel(const IdxT* __restrict__ crow, const IdxT* __restrict__ dst, long long num_dst,
                                    long long rows, long long fanout, const unsigned* __restrict__ dkey_sorted,
                                    long long* __restrict__ kcnt, int* __restrict__ longs, unsigned* __restrict__ nlong,
                                    long long* __restrict__ counts) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i > num_dst) return;
  if (i == num_dst) { kcnt[i] = 0; return; }
  const long long v = static_cast<long long>(dst[i]);
  bool valid = v >= 0 && v < rows;
  if (valid) {
    const unsigned u = static_cast<unsigned>(v);
    const long long lb = lower_bound(dkey_sorted, num_dst, u);   // first occurrence of u
    valid = !(lb + 1 < num_dst && dkey_sorted[lb + 1] == u);
  }
  long long k = 0;
  if (valid) {
    const long long deg = static_cast<long long>(crow[v + 1]) - static_cast<long long>(crow[v]);
    k = fanout < 0 ? deg : (deg < fanout ? deg : fanout);
    if (k > 0 && deg > kLongRow) longs[atomicAdd(nlong, 1u)] = static_cast<int>(i);
  } else {
    atomicAdd(reinterpret_cast<unsigned long long*>(&counts[2]), 1ull);
  }
  kcnt[i] = k;
}

// Slots the selection does not fill (all of them when the capacity is exceeded) hold the sentinel,
// so that the sort over `cap` ids places them last.
__global__ void sample_fill_kernel(const long long* __restrict__ slot, long long num_dst, long long cap,
                                   unsigned sentinel, unsigned* __restrict__ stage_col) {
  const long long total = slot[num_dst];
  const long long from = total > cap ? 0 : total;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long p = from + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; p < cap; p += stride)
    stage_col[p] = sentinel;
}

// Shared state of one group of G threads (a warp, or a CTA) sampling one row.
template <int G>
struct RowShared {
  unsigned hist[256];
  long long before, cnt;
  int bucket;
  int warp_eq[G / 32], warp_sel[G / 32];
};

template <int G>
__device__ __forceinline__ void group_sync() {
  if constexpr (G == 32) __syncwarp(); else __syncthreads();
}

// Exclusive prefix over the warps of the group of a per-warp count, and the group total.  G > 32.
template <int G>
__device__ __forceinline__ long long group_prefix(int* slots, int warp, int lane, int mine, long long* total) {
  if (lane == 0) slots[warp] = mine;
  __syncthreads();
  long long before = 0, all = 0;
#pragma unroll
  for (int w = 0; w < G / 32; ++w) {
    const int c = slots[w];
    before += w < warp ? c : 0;
    all += c;
  }
  *total = all;
  return before;
}

// Samples row v (entries [b, b + deg) of A) into stage slots [off, off + k), in ascending j.
// Uniform over the group: every thread calls it with the same arguments except `tid`.
template <int G, typename IdxT, typename VT>
__device__ void sample_row(RowShared<G>& sh, int tid, const IdxT* __restrict__ col, const VT* __restrict__ val,
                           long long b, long long deg, long long k, unsigned long long h0, long long cols,
                           long long off, unsigned* __restrict__ stage_col, VT* __restrict__ stage_val) {
  const int lane = tid & 31, warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  const bool all = k >= deg;
  // Selected: key < thr, or key == thr among the first `need` such entries (ascending j).
  unsigned long long thr = ~0ull;
  long long need = deg;
  if (!all) {
    unsigned long long prefix = 0, mask = 0;
    long long rem = k;   // entries still to take among those whose key matches `prefix` under `mask`
    for (int shift = 56; shift >= 0; shift -= 8) {
      for (int i = tid; i < 256; i += G) sh.hist[i] = 0;
      group_sync<G>();
      for (long long j = tid; j < deg; j += G) {
        const unsigned long long key = mix64(h0 + static_cast<unsigned long long>(j));
        if ((key & mask) == prefix) atomicAdd(&sh.hist[(key >> shift) & 255], 1u);
      }
      group_sync<G>();
      if (warp == 0) {
        unsigned c[8];
        long long s = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) { c[q] = sh.hist[lane * 8 + q]; s += c[q]; }
        long long incl = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const long long t = __shfl_up_sync(kFull, incl, o);
          if (lane >= o) incl += t;
        }
        const long long excl = incl - s;
        const unsigned hit = __ballot_sync(kFull, excl < rem && rem <= incl);
        if (lane == __ffs(hit) - 1) {
          long long before = excl;
          int q = 0;
          while (before + c[q] < rem) before += c[q++];
          sh.bucket = lane * 8 + q;
          sh.before = before;
          sh.cnt = c[q];
        }
      }
      group_sync<G>();
      const long long cnt = sh.cnt;
      rem -= sh.before;
      prefix |= static_cast<unsigned long long>(sh.bucket) << shift;
      mask |= 255ull << shift;
      group_sync<G>();   // sh is rewritten by the next pass
      if (rem == cnt) {  // the whole bucket is taken: every key up to its last value is selected
        thr = prefix | ~mask;
        break;
      }
      if (shift == 0) { thr = prefix; need = rem; }
    }
  }
  long long sel_before = 0, eq_before = 0;
  for (long long base = 0; base < deg; base += G) {
    const long long j = base + tid;
    const bool in = j < deg;
    bool sel = in;
    if (!all) {
      const unsigned long long key = in ? mix64(h0 + static_cast<unsigned long long>(j)) : 0ull;
      const bool eq = in && key == thr;
      const unsigned eqm = __ballot_sync(kFull, eq);
      long long eq_rank = eq_before + __popc(eqm & lt_mask), eq_total = __popc(eqm);
      if constexpr (G > 32) eq_rank += group_prefix<G>(sh.warp_eq, warp, lane, __popc(eqm), &eq_total);
      sel = in && (key < thr || (eq && eq_rank < need));
      eq_before += eq_total;
    }
    const unsigned selm = __ballot_sync(kFull, sel);
    long long pos = sel_before + __popc(selm & lt_mask), sel_total = __popc(selm);
    if constexpr (G > 32) pos += group_prefix<G>(sh.warp_sel, warp, lane, __popc(selm), &sel_total);
    if (sel) {
      const long long c = static_cast<long long>(col[b + j]);
      stage_col[off + pos] = static_cast<unsigned>(c >= 0 && c < cols ? c : cols);
      if (val != nullptr) stage_val[off + pos] = val[b + j];
    }
    sel_before += sel_total;
    group_sync<G>();   // warp_eq / warp_sel are rewritten by the next chunk
  }
}

template <typename IdxT, typename VT>
__global__ void __launch_bounds__(kSampleWarps * 32)
sample_rows_warp_kernel(const IdxT* __restrict__ crow, const IdxT* __restrict__ col, const VT* __restrict__ val,
                        long long cols, const IdxT* __restrict__ dst, long long num_dst,
                        const long long* __restrict__ slot, long long cap, unsigned long long seed,
                        unsigned* __restrict__ stage_col, VT* __restrict__ stage_val) {
  __shared__ RowShared<32> sh[kSampleWarps];
  if (slot[num_dst] > cap) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long step = static_cast<long long>(gridDim.x) * kSampleWarps;
  for (long long i = static_cast<long long>(blockIdx.x) * kSampleWarps + warp; i < num_dst; i += step) {
    const long long off = slot[i], k = slot[i + 1] - off;
    if (k == 0) continue;
    const long long v = static_cast<long long>(dst[i]);
    const long long b = static_cast<long long>(crow[v]), deg = static_cast<long long>(crow[v + 1]) - b;
    if (deg > kLongRow) continue;
    sample_row<32>(sh[warp], lane, col, val, b, deg, k, mix64(seed ^ static_cast<unsigned long long>(v)), cols, off,
                   stage_col, stage_val);
  }
}

template <typename IdxT, typename VT>
__global__ void __launch_bounds__(kLongThreads)
sample_long_rows_kernel(const IdxT* __restrict__ crow, const IdxT* __restrict__ col, const VT* __restrict__ val,
                        long long cols, const IdxT* __restrict__ dst, long long num_dst,
                        const long long* __restrict__ slot, long long cap, unsigned long long seed,
                        const int* __restrict__ longs, const unsigned* __restrict__ nlong,
                        unsigned* __restrict__ stage_col, VT* __restrict__ stage_val) {
  __shared__ RowShared<kLongThreads> sh;
  if (slot[num_dst] > cap) return;
  const unsigned n = *nlong;
  for (unsigned r = blockIdx.x; r < n; r += gridDim.x) {
    const long long i = longs[r];
    const long long off = slot[i], k = slot[i + 1] - off;
    const long long v = static_cast<long long>(dst[i]);
    const long long b = static_cast<long long>(crow[v]), deg = static_cast<long long>(crow[v + 1]) - b;
    sample_row<kLongThreads>(sh, threadIdx.x, col, val, b, deg, k, mix64(seed ^ static_cast<unsigned long long>(v)),
                             cols, off, stage_col, stage_val);
  }
}

// flag[p]: bit 0 = ids[p] is the first copy of a sampled id that is not a destination (a new
// source node), bit 32 = slot p holds a kept entry (column inside [0, cols)).  flag[cap] = 0.
__global__ void sample_flags_kernel(const unsigned* __restrict__ stage_col, const unsigned* __restrict__ ids,
                                    long long cap, const unsigned* __restrict__ dkey_sorted, long long num_dst,
                                    unsigned sentinel, long long* __restrict__ flag) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; p <= cap; p += stride) {
    if (p == cap) { flag[p] = 0; continue; }
    const unsigned u = ids[p];
    bool fresh = u != sentinel && (p == 0 || ids[p - 1] != u);
    if (fresh) {
      const long long lb = lower_bound(dkey_sorted, num_dst, u);
      fresh = !(lb < num_dst && dkey_sorted[lb] == u);
    }
    flag[p] = (fresh ? 1ll : 0ll) | (stage_col[p] != sentinel ? (1ll << 32) : 0ll);
  }
}

// Writes the block: kept entries compacted to their local ids, src_nodes, blk_crow and counts.
template <typename IdxT, typename VT>
__global__ void sample_emit_kernel(const IdxT* __restrict__ dst, long long num_dst, const long long* __restrict__ slot,
                                   long long cap, const unsigned* __restrict__ stage_col,
                                   const VT* __restrict__ stage_val, const unsigned* __restrict__ ids,
                                   const unsigned* __restrict__ dkey_sorted, const int* __restrict__ didx_sorted,
                                   const long long* __restrict__ flag, const long long* __restrict__ scan,
                                   unsigned sentinel, int* __restrict__ blk_crow, int* __restrict__ blk_col,
                                   VT* __restrict__ blk_val, IdxT* __restrict__ src_nodes, long long* __restrict__ counts) {
  const long long total = slot[num_dst];
  const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (total > cap) {   // outputs invalid: only the needed size is reported
    if (tid == 0) { counts[0] = total; counts[1] = 0; }
    return;
  }
  constexpr long long kLow = 0xffffffffll;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  const long long n = cap > num_dst + 1 ? cap : num_dst + 1;
  for (long long p = tid; p < n; p += stride) {
    if (p < cap) {
      const unsigned u = stage_col[p];
      if (u != sentinel) {
        const long long lb = lower_bound(dkey_sorted, num_dst, u);
        long long local;
        if (lb < num_dst && dkey_sorted[lb] == u) local = didx_sorted[lb];
        else local = num_dst + (scan[lower_bound(ids, cap, u)] & kLow);
        const long long q = scan[p] >> 32;
        blk_col[q] = static_cast<int>(local);
        if (blk_val != nullptr) blk_val[q] = stage_val[p];
      }
      if (flag[p] & 1) src_nodes[num_dst + (scan[p] & kLow)] = static_cast<IdxT>(ids[p]);
    }
    if (p < num_dst) src_nodes[p] = dst[p];
    if (p <= num_dst) blk_crow[p] = static_cast<int>(scan[slot[p]] >> 32);
    if (p == 0) {
      counts[0] = scan[cap] >> 32;
      counts[1] = num_dst + (scan[cap] & kLow);
    }
  }
}

struct SampleLayout {
  size_t hdr, dkey_in, dkey_out, didx_in, didx_out, kcnt, slot, longs, stage_col, ids, stage_val, flag, scan, cub_tmp,
      cub_bytes, total;
};

SampleLayout sample_layout(int64_t num_dst, int64_t cap) {
  SampleLayout L;
  const size_t nd = static_cast<size_t>(num_dst > 0 ? num_dst : 1), nc = static_cast<size_t>(cap > 0 ? cap : 1);
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t at = off; off += align_up(bytes, 256); return at; };
  L.hdr = take(256);
  L.dkey_in = take(nd * 4);
  L.dkey_out = take(nd * 4);
  L.didx_in = take(nd * 4);
  L.didx_out = take(nd * 4);
  L.kcnt = take((nd + 1) * 8);
  L.slot = take((nd + 1) * 8);
  L.longs = take(nd * 4);
  L.stage_col = take(nc * 4);
  L.ids = take(nc * 4);
  L.stage_val = take(nc * 4);
  L.flag = take((nc + 1) * 8);
  L.scan = take((nc + 1) * 8);
  // temporary storage of the widest key range (32 bits) bounds that of every narrower one
  size_t b1 = 0, b2 = 0, b3 = 0, b4 = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, b1, static_cast<const unsigned*>(nullptr), static_cast<unsigned*>(nullptr),
                                  static_cast<const int*>(nullptr), static_cast<int*>(nullptr), static_cast<int>(nd), 0, 32);
  cub::DeviceRadixSort::SortKeys(nullptr, b2, static_cast<const unsigned*>(nullptr), static_cast<unsigned*>(nullptr),
                                 static_cast<int>(nc), 0, 32);
  cub::DeviceScan::ExclusiveSum(nullptr, b3, static_cast<const long long*>(nullptr), static_cast<long long*>(nullptr),
                                static_cast<int>(nd + 1));
  cub::DeviceScan::ExclusiveSum(nullptr, b4, static_cast<const long long*>(nullptr), static_cast<long long*>(nullptr),
                                static_cast<int>(nc + 1));
  L.cub_bytes = b1;
  if (b2 > L.cub_bytes) L.cub_bytes = b2;
  if (b3 > L.cub_bytes) L.cub_bytes = b3;
  if (b4 > L.cub_bytes) L.cub_bytes = b4;
  L.cub_tmp = take(L.cub_bytes);
  L.total = off;
  return L;
}

template <typename IdxT, typename VT>
int sample_impl(const ofspmm_csr* A, const void* dst_v, int64_t num_dst, int64_t fanout, uint64_t seed, int64_t cap,
                void* blk_crow, void* blk_col, void* blk_val, void* src_nodes, int64_t* counts, void* ws,
                cudaStream_t stream) {
  const SampleLayout L = sample_layout(num_dst, cap);
  unsigned char* w = static_cast<unsigned char*>(ws);
  unsigned* nlong = reinterpret_cast<unsigned*>(w + L.hdr);
  unsigned* dkey_in = reinterpret_cast<unsigned*>(w + L.dkey_in);
  unsigned* dkey = reinterpret_cast<unsigned*>(w + L.dkey_out);
  int* didx_in = reinterpret_cast<int*>(w + L.didx_in);
  int* didx = reinterpret_cast<int*>(w + L.didx_out);
  long long* kcnt = reinterpret_cast<long long*>(w + L.kcnt);
  long long* slot = reinterpret_cast<long long*>(w + L.slot);
  int* longs = reinterpret_cast<int*>(w + L.longs);
  unsigned* stage_col = reinterpret_cast<unsigned*>(w + L.stage_col);
  unsigned* ids = reinterpret_cast<unsigned*>(w + L.ids);
  VT* stage_val = reinterpret_cast<VT*>(w + L.stage_val);
  long long* flag = reinterpret_cast<long long*>(w + L.flag);
  long long* scan = reinterpret_cast<long long*>(w + L.scan);
  void* tmp = w + L.cub_tmp;
  const IdxT* crow = static_cast<const IdxT*>(A->crow);
  const IdxT* col = static_cast<const IdxT*>(A->col);
  const VT* val = static_cast<const VT*>(A->val);
  const IdxT* dst = static_cast<const IdxT*>(dst_v);
  const long long rows = A->rows;
  const unsigned sentinel = static_cast<unsigned>(rows);
  const int bits = id_bits(rows);
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  const int grid = dev.sms * 8;
  auto blocks = [&](long long n, int threads) {
    const long long g = (n + threads - 1) / threads;
    return static_cast<unsigned>(g < 1 ? 1 : (g > grid ? grid : g));
  };

  OFSPMM_CUDA_OK(cudaMemsetAsync(counts, 0, 3 * sizeof(int64_t), stream));
  OFSPMM_CUDA_OK(cudaMemsetAsync(nlong, 0, sizeof(unsigned), stream));
  size_t cub_bytes = L.cub_bytes;
  if (num_dst > 0) {
    sample_dst_keys_kernel<IdxT><<<blocks(num_dst, 256), 256, 0, stream>>>(dst, num_dst, rows, dkey_in, didx_in);
    count_launch();
    OFSPMM_CUDA_OK(cub::DeviceRadixSort::SortPairs(tmp, cub_bytes, static_cast<const unsigned*>(dkey_in), dkey,
                                                   static_cast<const int*>(didx_in), didx, static_cast<int>(num_dst), 0,
                                                   bits, stream));
    count_launch(4);
  }
  sample_count_kernel<IdxT><<<static_cast<unsigned>((num_dst + 1 + 255) / 256), 256, 0, stream>>>(
      crow, dst, num_dst, rows, fanout, dkey, kcnt, longs, nlong, reinterpret_cast<long long*>(counts));
  count_launch();
  cub_bytes = L.cub_bytes;
  OFSPMM_CUDA_OK(cub::DeviceScan::ExclusiveSum(tmp, cub_bytes, static_cast<const long long*>(kcnt), slot,
                                               static_cast<int>(num_dst + 1), stream));
  count_launch(2);
  if (cap > 0) {
    sample_fill_kernel<<<blocks(cap, 256), 256, 0, stream>>>(slot, num_dst, cap, sentinel, stage_col);
    count_launch();
  }
  if (num_dst > 0) {
    const long long wblocks = (num_dst + kSampleWarps - 1) / kSampleWarps;
    const unsigned wgrid = static_cast<unsigned>(wblocks < dev.sms * 16 ? wblocks : dev.sms * 16);
    sample_rows_warp_kernel<IdxT, VT><<<wgrid, kSampleWarps * 32, 0, stream>>>(
        crow, col, val, A->cols, dst, num_dst, slot, cap, seed, stage_col, stage_val);
    const long long lgrid = num_dst < dev.sms * 2 ? num_dst : dev.sms * 2;
    sample_long_rows_kernel<IdxT, VT><<<static_cast<unsigned>(lgrid), kLongThreads, 0, stream>>>(
        crow, col, val, A->cols, dst, num_dst, slot, cap, seed, longs, nlong, stage_col, stage_val);
    count_launch(2);
  }
  if (cap > 0) {
    cub_bytes = L.cub_bytes;
    OFSPMM_CUDA_OK(cub::DeviceRadixSort::SortKeys(tmp, cub_bytes, static_cast<const unsigned*>(stage_col), ids,
                                                  static_cast<int>(cap), 0, bits, stream));
    count_launch(4);
  }
  sample_flags_kernel<<<blocks(cap + 1, 256), 256, 0, stream>>>(stage_col, ids, cap, dkey, num_dst, sentinel, flag);
  count_launch();
  cub_bytes = L.cub_bytes;
  OFSPMM_CUDA_OK(cub::DeviceScan::ExclusiveSum(tmp, cub_bytes, static_cast<const long long*>(flag), scan,
                                               static_cast<int>(cap + 1), stream));
  count_launch(2);
  sample_emit_kernel<IdxT, VT><<<blocks(cap > num_dst + 1 ? cap : num_dst + 1, 256), 256, 0, stream>>>(
      dst, num_dst, slot, cap, stage_col, stage_val, ids, dkey, didx, flag, scan, sentinel,
      static_cast<int*>(blk_crow), static_cast<int*>(blk_col), static_cast<VT*>(blk_val), static_cast<IdxT*>(src_nodes),
      reinterpret_cast<long long*>(counts));
  count_launch();
  OFSPMM_CUDA_OK(cudaGetLastError());
  return OFSPMM_OK;
}

template <typename IdxT>
int sample_by_val(const ofspmm_csr* A, const void* dst, int64_t num_dst, int64_t fanout, uint64_t seed, int64_t cap,
                  void* blk_crow, void* blk_col, void* blk_val, void* src_nodes, int64_t* counts, void* ws,
                  cudaStream_t stream) {
  // values are copied bit for bit: fp32 as 32-bit, bf16 as 16-bit words
  if (A->val_dtype == OFSPMM_DTYPE_FLOAT)
    return sample_impl<IdxT, uint32_t>(A, dst, num_dst, fanout, seed, cap, blk_crow, blk_col, blk_val, src_nodes, counts, ws, stream);
  if (A->val_dtype == OFSPMM_DTYPE_BFLOAT16)
    return sample_impl<IdxT, uint16_t>(A, dst, num_dst, fanout, seed, cap, blk_crow, blk_col, blk_val, src_nodes, counts, ws, stream);
  return sample_impl<IdxT, uint8_t>(A, dst, num_dst, fanout, seed, cap, blk_crow, blk_col, nullptr, src_nodes, counts, ws, stream);
}

}  // namespace

size_t sample_neighbors_workspace_bytes(int64_t num_dst, int64_t cap) { return sample_layout(num_dst, cap).total; }

int launch_sample_neighbors(const ofspmm_csr* A, const void* dst, int64_t num_dst, int64_t fanout, uint64_t seed,
                            int64_t cap, void* blk_crow, void* blk_col, void* blk_val, void* src_nodes, int64_t* counts,
                            void* ws, cudaStream_t stream) {
  if (A->idx_dtype == OFSPMM_DTYPE_INT32)
    return sample_by_val<int32_t>(A, dst, num_dst, fanout, seed, cap, blk_crow, blk_col, blk_val, src_nodes, counts, ws, stream);
  return sample_by_val<int64_t>(A, dst, num_dst, fanout, seed, cap, blk_crow, blk_col, blk_val, src_nodes, counts, ws, stream);
}

}  // namespace ofspmm
