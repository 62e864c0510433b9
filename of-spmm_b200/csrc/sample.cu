// sample.cu — device neighbour sampling (DESIGN.md §3.8): for each destination v, the k entries of
// row v with the smallest (key, j), then a relabel of the sampled columns into a bipartite block
// (DGL's block convention: the destinations come first in src_nodes, then the other sampled ids in
// ascending order).  Uniform: k = min(deg, fanout), key = x = mix(mix(seed ^ v) + j) (splitmix64);
// weighted: k = min(npos, fanout), key = bits(neglog(U(x)) / w_j), all ones for an ineligible weight
// (sample_key.h); with replacement: k = fanout independent draws j_t = mulhi(x(seed, v, t), deg).
// Edge exclusion (OFSPMM_SAMPLE_EXCLUDE) makes the excluded positions ineligible: the count, npos,
// select and draw kernels take the list as a trailing argument `ex...`, empty without the flag, so
// that the kernels of the calls without it are unchanged.
//   count   one thread per destination: validity (range, repeats found in the sorted ids), k, and a
//           list of the rows long enough for a whole CTA;
//   npos    weighted only: eligible entries per row, one warp per row (one CTA per long row);
//           k = min(npos, fanout);
//   select  one warp per destination (one CTA per long row): radix selection of the k-th smallest
//           key over re-computed keys, 8 bits per pass, stopping as soon as the bucket holding the
//           k-th key is taken whole; then one pass that emits the selected entries in ascending j
//           (ballot compaction), loading col / val for those only.  A row with deg <= k is copied.
//   draw    with replacement: one warp per destination, the draws in order t, col / val loaded at
//           the drawn positions only.
//   relabel radix sort of the sampled ids (cub, as the transpose does), unique / not-a-destination
//           flags, one scan that also compacts away the out-of-range columns, and a binary search
//           per kept entry for its local id.
// Everything the kernels address is sized by (num_dst, cap), never by A's rows.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "bsearch.cuh"
#include "launch.cuh"
#include "sample_key.h"

namespace ofspmm {

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kSampleWarps = 8;         // warps per CTA of the warp-per-row kernel
constexpr int kLongThreads = 512;       // threads per CTA of the long-row kernel
constexpr long long kLongRow = 4096;    // rows longer than this are sampled by a whole CTA

enum SampleMode { kUniform, kWeighted, kReplace };

// Keys of the selection: position j of the row that starts at entry b of A.
struct UniformKey {
  unsigned long long h0;
  __device__ __forceinline__ UniformKey(unsigned long long seed, long long v, long long, const void*)
      : h0(sk_mix64(seed ^ static_cast<unsigned long long>(v))) {}
  __device__ __forceinline__ unsigned long long operator()(long long j) const {
    return sk_mix64(h0 + static_cast<unsigned long long>(j));
  }
  __device__ __forceinline__ bool excluded(long long) const { return false; }
};

// A weight widened exactly to fp64: fp32 bits, or bf16 bits (the high half of an fp32).
__device__ __forceinline__ double widen(uint32_t b) { return static_cast<double>(__uint_as_float(b)); }
__device__ __forceinline__ double widen(uint16_t b) { return static_cast<double>(__uint_as_float(static_cast<uint32_t>(b) << 16)); }

// PT: uint32_t (fp32 weights) or uint16_t (bf16 weights).  The weight is re-read per evaluation.
template <typename PT>
struct WeightedKey {
  unsigned long long h0;
  const PT* p;
  __device__ __forceinline__ WeightedKey(unsigned long long seed, long long v, long long b, const void* prob)
      : h0(sk_mix64(seed ^ static_cast<unsigned long long>(v))), p(static_cast<const PT*>(prob) + b) {}
  __device__ __forceinline__ unsigned long long operator()(long long j) const {
    return sk_weighted_key(sk_mix64(h0 + static_cast<unsigned long long>(j)), widen(p[j]));
  }
  __device__ __forceinline__ bool excluded(long long) const { return false; }
};

// OFSPMM_SAMPLE_EXCLUDE: `n` strictly ascending positions in A.
template <typename IdxT>
struct ExcludeList {
  const IdxT* pos;
  long long n;
};

// The excluded positions of one row: none without an exclusion list (every member folds away).
struct NoExcludedRow {
  __device__ __forceinline__ long long count() const { return 0; }
  __device__ __forceinline__ bool has(long long) const { return false; }
};

// pos[0, cnt): the excluded positions inside the row [b, b + deg) of A, ascending.
template <typename IdxT>
struct ExcludedRow {
  const IdxT* pos;
  long long cnt, b, deg;
  // Excluded entries of the row, at most deg (a list with repeats is not strictly ascending: the
  // blocks are unspecified, but no row takes more than it has).
  __device__ __forceinline__ long long count() const { return cnt < deg ? cnt : deg; }
  // Position e of A is excluded: a search of a usually empty range.
  __device__ __forceinline__ bool has(long long e) const {
    const long long q = lower_bound(pos, cnt, static_cast<IdxT>(e));
    return q < cnt && static_cast<long long>(pos[q]) == e;
  }
  // Offset in the row of its r-th eligible entry (ascending): r plus the excluded positions passed.
  __device__ __forceinline__ long long position(long long r) const {
    long long j = r;
    for (long long q = 0; q < cnt && static_cast<long long>(pos[q]) <= b + j; ++q) ++j;
    return j;
  }
};

__device__ __forceinline__ NoExcludedRow excluded_row(long long, long long) { return {}; }

template <typename IdxT>
__device__ __forceinline__ ExcludedRow<IdxT> excluded_row(long long b, long long deg, const ExcludeList<IdxT>& ex) {
  const long long lo = lower_bound(ex.pos, ex.n, static_cast<IdxT>(b));
  const long long hi = lower_bound(ex.pos, ex.n, static_cast<IdxT>(b + deg));
  return {ex.pos + lo, hi - lo, b, deg};
}

// A selection key whose excluded entries get the key all ones and no place in the tie rank.
template <typename Key, typename IdxT>
struct ExcludedKey {
  Key key;
  ExcludedRow<IdxT> row;
  __device__ __forceinline__ unsigned long long operator()(long long j) const { return excluded(j) ? ~0ull : key(j); }
  __device__ __forceinline__ bool excluded(long long j) const { return row.cnt != 0 && row.has(row.b + j); }
};

// Offset in the row of the draw x: mulhi(x, deg); with an exclusion list the mulhi(x, n_e)-th
// eligible entry.
__device__ __forceinline__ long long draw_offset(unsigned long long x, long long deg, const NoExcludedRow&) {
  return static_cast<long long>(__umul64hi(x, static_cast<unsigned long long>(deg)));
}

template <typename IdxT>
__device__ __forceinline__ long long draw_offset(unsigned long long x, long long deg, const ExcludedRow<IdxT>& row) {
  return row.position(static_cast<long long>(__umul64hi(x, static_cast<unsigned long long>(deg - row.count()))));
}

template <typename Key>
__device__ __forceinline__ Key with_exclusion(const Key& key, const NoExcludedRow&) { return key; }

template <typename Key, typename IdxT>
__device__ __forceinline__ ExcludedKey<Key, IdxT> with_exclusion(const Key& key, const ExcludedRow<IdxT>& row) {
  return {key, row};
}

// Bits of a sort key that holds ids in [0, rows] (rows itself is the "no id" sentinel).
int id_bits(long long rows) {
  int b = 1;
  while (b < 32 && (1ll << b) <= rows) ++b;
  return b;
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
// once); kcnt[num_dst] = 0 so that the exclusive scan ends in the total.  Weighted: k from deg is
// only an upper bound, which sample_npos / sample_npos_long turn into min(npos, fanout).  With an
// exclusion list the row's excluded entries are not counted: k from n_e = deg - excluded.
template <typename IdxT, typename... Ex>
__global__ void sample_count_kernel(const IdxT* __restrict__ crow, const IdxT* __restrict__ dst, long long num_dst,
                                    long long rows, long long fanout, int mode, const unsigned* __restrict__ dkey_sorted,
                                    long long* __restrict__ kcnt, int* __restrict__ longs, unsigned* __restrict__ nlong,
                                    long long* __restrict__ counts, Ex... ex) {
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
    const long long ne = deg - excluded_row(static_cast<long long>(crow[v]), deg, ex...).count();
    if (mode == kReplace) {
      k = ne > 0 ? fanout : 0;   // fanout >= 0: draws need no selection, hence no long-row list
    } else {
      k = fanout < 0 ? ne : (ne < fanout ? ne : fanout);
      if (k > 0 && deg > kLongRow) longs[atomicAdd(nlong, 1u)] = static_cast<int>(i);
    }
  } else {
    atomicAdd(reinterpret_cast<unsigned long long*>(&counts[2]), 1ull);
  }
  kcnt[i] = k;
}

// Weighted: kcnt[i] = min(npos, fanout) (npos for fanout -1) of the listed long rows, one CTA per
// row, as their selection runs.
template <typename IdxT, typename PT, typename... Ex>
__global__ void __launch_bounds__(kLongThreads)
sample_npos_long_kernel(const IdxT* __restrict__ crow, const IdxT* __restrict__ dst, long long fanout,
                        const PT* __restrict__ prob, const int* __restrict__ longs, const unsigned* __restrict__ nlong,
                        long long* __restrict__ kcnt, Ex... ex) {
  __shared__ unsigned warp_cnt[kLongThreads / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned n = *nlong;
  for (unsigned r = blockIdx.x; r < n; r += gridDim.x) {
    const long long i = longs[r];
    const long long v = static_cast<long long>(dst[i]);
    const long long b = static_cast<long long>(crow[v]), deg = static_cast<long long>(crow[v + 1]) - b;
    const auto xr = excluded_row(b, deg, ex...);
    unsigned c = 0;
    for (long long j = threadIdx.x; j < deg; j += kLongThreads)
      c += sk_eligible(widen(prob[b + j])) && !xr.has(b + j) ? 1u : 0u;
    c = __reduce_add_sync(kFull, c);
    if (lane == 0) warp_cnt[warp] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
      long long npos = 0;
#pragma unroll
      for (int w = 0; w < kLongThreads / 32; ++w) npos += warp_cnt[w];
      kcnt[i] = fanout >= 0 && npos > fanout ? fanout : npos;
    }
    __syncthreads();   // warp_cnt is rewritten for the next row
  }
}

// Weighted: kcnt[i] = min(npos, fanout) (npos for fanout -1), one warp per destination of at most
// kLongRow entries; the longer ones are sample_npos_long's.
template <typename IdxT, typename PT, typename... Ex>
__global__ void __launch_bounds__(kSampleWarps * 32)
sample_npos_kernel(const IdxT* __restrict__ crow, const IdxT* __restrict__ dst, long long num_dst, long long fanout,
                   const PT* __restrict__ prob, long long* __restrict__ kcnt, Ex... ex) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long step = static_cast<long long>(gridDim.x) * kSampleWarps;
  for (long long i = static_cast<long long>(blockIdx.x) * kSampleWarps + warp; i < num_dst; i += step) {
    if (kcnt[i] == 0) continue;   // invalid, empty row or fanout 0
    const long long v = static_cast<long long>(dst[i]);
    const long long b = static_cast<long long>(crow[v]), deg = static_cast<long long>(crow[v + 1]) - b;
    if (deg > kLongRow) continue;
    const auto xr = excluded_row(b, deg, ex...);
    unsigned c = 0;
    for (long long j = lane; j < deg; j += 32) c += sk_eligible(widen(prob[b + j])) && !xr.has(b + j) ? 1u : 0u;
    const long long npos = __reduce_add_sync(kFull, c);
    if (lane == 0) kcnt[i] = fanout >= 0 && npos > fanout ? fanout : npos;
  }
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

// Samples row v (entries [b, b + deg) of A) into stage slots [off, off + k), in ascending j, by the
// keys key(j).  Uniform over the group: every thread calls it with the same arguments except `tid`.
// stage_eid (may be null) receives the positions b + j in A.  An entry key_of.excluded(j) is never
// selected: k counts eligible entries only, its key is all ones, and it takes no place in the ties.
template <int G, typename IdxT, typename VT, typename Key>
__device__ void sample_row(RowShared<G>& sh, int tid, const IdxT* __restrict__ col, const VT* __restrict__ val,
                           long long b, long long deg, long long k, const Key& key_of, long long cols,
                           long long off, unsigned* __restrict__ stage_col, VT* __restrict__ stage_val,
                           long long* __restrict__ stage_eid) {
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
        const unsigned long long key = key_of(j);
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
      const unsigned long long key = in ? key_of(j) : 0ull;
      const bool eq = in && key == thr && !key_of.excluded(j);
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
      if (stage_eid != nullptr) stage_eid[off + pos] = b + j;
    }
    sel_before += sel_total;
    group_sync<G>();   // warp_eq / warp_sel are rewritten by the next chunk
  }
}

template <typename IdxT, typename VT, typename Key, typename... Ex>
__global__ void __launch_bounds__(kSampleWarps * 32)
sample_rows_warp_kernel(const IdxT* __restrict__ crow, const IdxT* __restrict__ col, const VT* __restrict__ val,
                        long long cols, const IdxT* __restrict__ dst, long long num_dst,
                        const long long* __restrict__ slot, long long cap, unsigned long long seed,
                        const void* __restrict__ prob, unsigned* __restrict__ stage_col, VT* __restrict__ stage_val,
                        long long* __restrict__ stage_eid, Ex... ex) {
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
    sample_row<32>(sh[warp], lane, col, val, b, deg, k, with_exclusion(Key(seed, v, b, prob), excluded_row(b, deg, ex...)),
                   cols, off, stage_col, stage_val, stage_eid);
  }
}

template <typename IdxT, typename VT, typename Key, typename... Ex>
__global__ void __launch_bounds__(kLongThreads)
sample_long_rows_kernel(const IdxT* __restrict__ crow, const IdxT* __restrict__ col, const VT* __restrict__ val,
                        long long cols, const IdxT* __restrict__ dst, long long num_dst,
                        const long long* __restrict__ slot, long long cap, unsigned long long seed,
                        const void* __restrict__ prob, const int* __restrict__ longs, const unsigned* __restrict__ nlong,
                        unsigned* __restrict__ stage_col, VT* __restrict__ stage_val, long long* __restrict__ stage_eid,
                        Ex... ex) {
  __shared__ RowShared<kLongThreads> sh;
  if (slot[num_dst] > cap) return;
  const unsigned n = *nlong;
  for (unsigned r = blockIdx.x; r < n; r += gridDim.x) {
    const long long i = longs[r];
    const long long off = slot[i], k = slot[i + 1] - off;
    if (k == 0) continue;   // weighted: no eligible entry
    const long long v = static_cast<long long>(dst[i]);
    const long long b = static_cast<long long>(crow[v]), deg = static_cast<long long>(crow[v + 1]) - b;
    sample_row<kLongThreads>(sh, threadIdx.x, col, val, b, deg, k,
                             with_exclusion(Key(seed, v, b, prob), excluded_row(b, deg, ex...)), cols, off, stage_col,
                             stage_val, stage_eid);
  }
}

// With replacement: draw t of destination v takes position j_t = mulhi(x(seed, v, t), deg) into
// slot off + t; one warp per destination, col / val read at the drawn positions only.  With an
// exclusion list: the r_t-th eligible position, r_t = mulhi(x(seed, v, t), n_e).
template <typename IdxT, typename VT, typename... Ex>
__global__ void __launch_bounds__(kSampleWarps * 32)
sample_draw_kernel(const IdxT* __restrict__ crow, const IdxT* __restrict__ col, const VT* __restrict__ val,
                   long long cols, const IdxT* __restrict__ dst, long long num_dst, const long long* __restrict__ slot,
                   long long cap, unsigned long long seed, unsigned* __restrict__ stage_col,
                   VT* __restrict__ stage_val, long long* __restrict__ stage_eid, Ex... ex) {
  if (slot[num_dst] > cap) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long step = static_cast<long long>(gridDim.x) * kSampleWarps;
  for (long long i = static_cast<long long>(blockIdx.x) * kSampleWarps + warp; i < num_dst; i += step) {
    const long long off = slot[i], k = slot[i + 1] - off;
    if (k == 0) continue;
    const long long v = static_cast<long long>(dst[i]);
    const long long b = static_cast<long long>(crow[v]), deg = static_cast<long long>(crow[v + 1]) - b;
    const UniformKey x(seed, v, b, nullptr);
    const auto xr = excluded_row(b, deg, ex...);
    for (long long t = lane; t < k; t += 32) {
      const long long e = b + draw_offset(x(t), deg, xr);
      const long long c = static_cast<long long>(col[e]);
      stage_col[off + t] = static_cast<unsigned>(c >= 0 && c < cols ? c : cols);
      if (val != nullptr) stage_val[off + t] = val[e];
      if (stage_eid != nullptr) stage_eid[off + t] = e;
    }
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
                                   const VT* __restrict__ stage_val, const long long* __restrict__ stage_eid,
                                   const unsigned* __restrict__ ids,
                                   const unsigned* __restrict__ dkey_sorted, const int* __restrict__ didx_sorted,
                                   const long long* __restrict__ flag, const long long* __restrict__ scan,
                                   unsigned sentinel, int* __restrict__ blk_crow, int* __restrict__ blk_col,
                                   VT* __restrict__ blk_val, IdxT* __restrict__ blk_eid, IdxT* __restrict__ src_nodes,
                                   long long* __restrict__ counts) {
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
        if (blk_eid != nullptr) blk_eid[q] = static_cast<IdxT>(stage_eid[p]);
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
      cub_bytes, stage_eid, total;
};

SampleLayout sample_layout(int64_t num_dst, int64_t cap, bool edge_ids) {
  SampleLayout L;
  const size_t nd = static_cast<size_t>(num_dst > 0 ? num_dst : 1), nc = static_cast<size_t>(cap > 0 ? cap : 1);
  Carve c;
  L.hdr = c.take(256);
  L.dkey_in = c.take(nd * 4);
  L.dkey_out = c.take(nd * 4);
  L.didx_in = c.take(nd * 4);
  L.didx_out = c.take(nd * 4);
  L.kcnt = c.take((nd + 1) * 8);
  L.slot = c.take((nd + 1) * 8);
  L.longs = c.take(nd * 4);
  L.stage_col = c.take(nc * 4);
  L.ids = c.take(nc * 4);
  L.stage_val = c.take(nc * 4);
  L.flag = c.take((nc + 1) * 8);
  L.scan = c.take((nc + 1) * 8);
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
  L.cub_tmp = c.take(L.cub_bytes);
  L.stage_eid = edge_ids ? c.take(nc * 8) : 0;   // last, so that the layout without it is unchanged
  L.total = c.total;
  return L;
}

// The sampling mode of a call, its weights and its exclusion list (validated options; NULL
// options: uniform, nothing excluded).
struct SampleCall {
  int mode;
  const void* prob;
  int prob_dtype;
  const void* exclude;
  int64_t num_exclude;
};

// ex...: an ExcludeList<IdxT> for a call with a non-empty exclusion list, else nothing.
template <typename IdxT, typename VT, typename... Ex>
int sample_impl(const ofspmm_csr* A, const SampleCall& m, const void* dst_v, int64_t num_dst, int64_t fanout,
                uint64_t seed, int64_t cap, void* blk_crow, void* blk_col, void* blk_val, void* blk_eid,
                void* src_nodes, int64_t* counts, void* ws, cudaStream_t stream, Ex... ex) {
  const SampleLayout L = sample_layout(num_dst, cap, blk_eid != nullptr);
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
  long long* stage_eid = blk_eid != nullptr ? reinterpret_cast<long long*>(w + L.stage_eid) : nullptr;
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
  auto blocks = [&](long long n) { return grid_for(n, 256, dev.sms * 8, dev.sms); };
  const long long wblocks = (num_dst + kSampleWarps - 1) / kSampleWarps;
  const unsigned wgrid = static_cast<unsigned>(wblocks < dev.sms * 16 ? wblocks : dev.sms * 16);

  OFSPMM_CUDA_OK(cudaMemsetAsync(counts, 0, 3 * sizeof(int64_t), stream));
  OFSPMM_CUDA_OK(cudaMemsetAsync(nlong, 0, sizeof(unsigned), stream));
  size_t cub_bytes = L.cub_bytes;
  if (num_dst > 0) {
    sample_dst_keys_kernel<IdxT><<<blocks(num_dst), 256, 0, stream>>>(dst, num_dst, rows, dkey_in, didx_in);
    count_launch();
    OFSPMM_CUDA_OK(cub::DeviceRadixSort::SortPairs(tmp, cub_bytes, static_cast<const unsigned*>(dkey_in), dkey,
                                                   static_cast<const int*>(didx_in), didx, static_cast<int>(num_dst), 0,
                                                   bits, stream));
    count_launch(4);
  }
  sample_count_kernel<IdxT, Ex...><<<static_cast<unsigned>((num_dst + 1 + 255) / 256), 256, 0, stream>>>(
      crow, dst, num_dst, rows, fanout, m.mode, dkey, kcnt, longs, nlong, reinterpret_cast<long long*>(counts), ex...);
  count_launch();
  // f(Tag<PT>{}) for the weights' bit type: fp32 or bf16 words
  auto by_prob = [&](auto&& f) { m.prob_dtype == OFSPMM_DTYPE_FLOAT ? f(Tag<uint32_t>{}) : f(Tag<uint16_t>{}); };
  if (m.mode == kWeighted && num_dst > 0) {
    by_prob([&](auto pt) {   // k = min(npos, fanout)
      using PT = typename decltype(pt)::type;
      const PT* prob = static_cast<const PT*>(m.prob);
      const long long lgrid = num_dst < dev.sms * 2 ? num_dst : dev.sms * 2;
      sample_npos_long_kernel<IdxT, PT, Ex...><<<static_cast<unsigned>(lgrid), kLongThreads, 0, stream>>>(
          crow, dst, fanout, prob, longs, nlong, kcnt, ex...);
      sample_npos_kernel<IdxT, PT, Ex...><<<wgrid, kSampleWarps * 32, 0, stream>>>(crow, dst, num_dst, fanout, prob, kcnt,
                                                                           ex...);
      count_launch(2);
    });
  }
  auto select = [&](auto key) {
    using Key = typename decltype(key)::type;
    sample_rows_warp_kernel<IdxT, VT, Key, Ex...><<<wgrid, kSampleWarps * 32, 0, stream>>>(
        crow, col, val, A->cols, dst, num_dst, slot, cap, seed, m.prob, stage_col, stage_val, stage_eid, ex...);
    const long long lgrid = num_dst < dev.sms * 2 ? num_dst : dev.sms * 2;
    sample_long_rows_kernel<IdxT, VT, Key, Ex...><<<static_cast<unsigned>(lgrid), kLongThreads, 0, stream>>>(
        crow, col, val, A->cols, dst, num_dst, slot, cap, seed, m.prob, longs, nlong, stage_col, stage_val, stage_eid,
        ex...);
    count_launch(2);
  };
  cub_bytes = L.cub_bytes;
  OFSPMM_CUDA_OK(cub::DeviceScan::ExclusiveSum(tmp, cub_bytes, static_cast<const long long*>(kcnt), slot,
                                               static_cast<int>(num_dst + 1), stream));
  count_launch(2);
  if (cap > 0) {
    sample_fill_kernel<<<blocks(cap), 256, 0, stream>>>(slot, num_dst, cap, sentinel, stage_col);
    count_launch();
  }
  if (num_dst > 0) {
    if (m.mode == kReplace) {
      sample_draw_kernel<IdxT, VT, Ex...><<<wgrid, kSampleWarps * 32, 0, stream>>>(
          crow, col, val, A->cols, dst, num_dst, slot, cap, seed, stage_col, stage_val, stage_eid, ex...);
      count_launch();
    } else if (m.mode == kWeighted) {
      by_prob([&](auto pt) { select(Tag<WeightedKey<typename decltype(pt)::type>>{}); });
    } else {
      select(Tag<UniformKey>{});
    }
  }
  if (cap > 0) {
    cub_bytes = L.cub_bytes;
    OFSPMM_CUDA_OK(cub::DeviceRadixSort::SortKeys(tmp, cub_bytes, static_cast<const unsigned*>(stage_col), ids,
                                                  static_cast<int>(cap), 0, bits, stream));
    count_launch(4);
  }
  sample_flags_kernel<<<blocks(cap + 1), 256, 0, stream>>>(stage_col, ids, cap, dkey, num_dst, sentinel, flag);
  count_launch();
  cub_bytes = L.cub_bytes;
  OFSPMM_CUDA_OK(cub::DeviceScan::ExclusiveSum(tmp, cub_bytes, static_cast<const long long*>(flag), scan,
                                               static_cast<int>(cap + 1), stream));
  count_launch(2);
  sample_emit_kernel<IdxT, VT><<<blocks(cap > num_dst + 1 ? cap : num_dst + 1), 256, 0, stream>>>(
      dst, num_dst, slot, cap, stage_col, stage_val, stage_eid, ids, dkey, didx, flag, scan, sentinel,
      static_cast<int*>(blk_crow), static_cast<int*>(blk_col), static_cast<VT*>(blk_val), static_cast<IdxT*>(blk_eid),
      static_cast<IdxT*>(src_nodes), reinterpret_cast<long long*>(counts));
  return launched();
}

}  // namespace

size_t sample_neighbors_workspace_bytes(int64_t num_dst, int64_t cap, bool edge_ids) {
  return sample_layout(num_dst, cap, edge_ids).total;
}

int launch_sample_neighbors(const ofspmm_csr* A, const ofspmm_sample_opts* opts, const void* dst, int64_t num_dst,
                            int64_t fanout, uint64_t seed, int64_t cap, void* blk_crow, void* blk_col, void* blk_val,
                            void* blk_eid, void* src_nodes, int64_t* counts, void* ws, cudaStream_t stream) {
  SampleCall m{kUniform, nullptr, 0, nullptr, 0};
  if (opts != nullptr && opts->prob != nullptr) m = {kWeighted, opts->prob, opts->prob_dtype, nullptr, 0};
  // fanout -1 with replacement is every entry once: the same block as without replacement
  else if (opts != nullptr && (opts->flags & OFSPMM_SAMPLE_REPLACE) && fanout >= 0) m.mode = kReplace;
  if (opts != nullptr && (opts->flags & OFSPMM_SAMPLE_EXCLUDE)) {
    m.exclude = opts->exclude;
    m.num_exclude = opts->num_exclude;
  }
  return dispatch_idx(A->idx_dtype, [&](auto idx) {
    using IdxT = typename decltype(idx)::type;
    // an empty exclusion list is the call without one: the same kernels
    auto run = [&](auto vt, void* bval, auto... ex) {
      return sample_impl<IdxT, typename decltype(vt)::type>(A, m, dst, num_dst, fanout, seed, cap, blk_crow, blk_col,
                                                            bval, blk_eid, src_nodes, counts, ws, stream, ex...);
    };
    auto run_ex = [&](auto vt, void* bval) {
      return m.num_exclude > 0 ? run(vt, bval, ExcludeList<IdxT>{static_cast<const IdxT*>(m.exclude), m.num_exclude})
                               : run(vt, bval);
    };
    // values are copied bit for bit: fp32 as 32-bit, bf16 as 16-bit words; a pattern matrix has none
    if (A->val_dtype == OFSPMM_VAL_UNIT) return run_ex(Tag<uint8_t>{}, nullptr);
    return dispatch_dense(A->val_dtype, [&](auto vt) {
      using VT = std::conditional_t<sizeof(typename decltype(vt)::type) == 4, uint32_t, uint16_t>;
      return run_ex(Tag<VT>{}, blk_val);
    });
  });
}

}  // namespace ofspmm
