// exchange.cu — row-exchange kernels of the multi-GPU path (SURVEY.md §8e) and the value re-gather
// of the cached-transpose backward.
//
// In the needed-rows exchange every rank keeps its shard of the dense operand in symmetric (peer
// mapped) memory; a rank PULLS exactly the B rows its row block touches straight out of the
// owners' HBM over NVLink / NVSwitch, and the dual for A^T·dY: the owner of a dB shard reads the
// peers' published partial rows and adds them in rank order (the rows of one list are distinct,
// so no atomics and a fixed summation order).  The reference instead materialises the whole
// operand on every rank with a blocking all-gather before the op is even issued
// (oneflow/core/boxing/ccl_boxing_function.cpp:105-124,183-197).
//
// Two generations live here:
//   * gather_rows / scatter_add_rows (+ the bf16 -> fp32 scatter, cast): one list, one peer per
//     launch, ordered by the caller (device barriers).  Building blocks with bit-exact tests; the
//     gloo emulation of the CPU tests has their semantics.
//   * signal_peers / pull_rows_tma / pull_rows_multi / combine_rows_multi (second half of the
//     file): the product path on NCCL groups.  ONE launch serves all peers; every segment spins
//     (ld.acquire.sys) on its owner's epoch flag, written by signal_peers_kernel with a release at
//     system scope after the owner's producing kernel — no host sync, no barrier kernel, no NCCL.
//     pull_rows_tma_kernel moves each row with a TMA bulk copy from PEER memory into a 5-stage
//     shared-memory ring and drains each stage with one bulk store: enough bytes in flight to cover
//     the ~2-3 us NVLink round trip with 64 one-warp CTAs, which fit into the CTA slot the
//     overlapped SpMM leaves free (ofspmm_opts.reserve_ctas_per_sm).
//
// Peer loads see ~2 us of latency: the register kernels keep UNROLL independent 16-byte units in
// flight per thread, and every grid is capped (`max_ctas`) so the copy shares the GPU with the
// SpMM kernel it overlaps.
#include "launch.cuh"

namespace ofspmm {

namespace {

constexpr int kThreads = 512;
constexpr int kUnroll = 4;

__device__ __forceinline__ uint4 ld_peer16(const void* p) {
  // plain (coherent) load: the source may live in a peer GPU's memory and is rewritten every step
  uint4 v;
  asm volatile("ld.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}

template <typename IdxT>
__device__ __forceinline__ long long list_at(const IdxT* list, long long i, long long off) {
  return list == nullptr ? i : static_cast<long long>(list[i]) - off;
}

// dst[i, :] = src[list[i] - off, :]; rows are `units` 16-byte units wide.
template <typename IdxT>
__global__ void __launch_bounds__(kThreads) gather_rows_kernel(
    char* __restrict__ dst, long long dst_stride, const char* __restrict__ src, long long src_stride,
    const IdxT* __restrict__ list, long long off, long long count, int units) {
  const long long total = count * units;
  const long long stride = static_cast<long long>(gridDim.x) * kThreads;
  long long u = static_cast<long long>(blockIdx.x) * kThreads + threadIdx.x;
  for (; u + (kUnroll - 1) * stride < total; u += kUnroll * stride) {
    uint4 v[kUnroll];
    long long drow[kUnroll];
    int c[kUnroll];
#pragma unroll
    for (int k = 0; k < kUnroll; ++k) {
      const long long uu = u + k * stride;
      drow[k] = uu / units;
      c[k] = static_cast<int>(uu - drow[k] * units);
      v[k] = ld_peer16(src + list_at(list, drow[k], off) * src_stride + c[k] * 16);
    }
#pragma unroll
    for (int k = 0; k < kUnroll; ++k)
      *reinterpret_cast<uint4*>(dst + drow[k] * dst_stride + c[k] * 16) = v[k];
  }
  for (; u < total; u += stride) {
    const long long r = u / units;
    const int c = static_cast<int>(u - r * units);
    *reinterpret_cast<uint4*>(dst + r * dst_stride + c * 16) = ld_peer16(src + list_at(list, r, off) * src_stride + c * 16);
  }
}

// element-wise fallback for rows that are not a whole number of aligned 16-byte units
template <typename IdxT, typename DT>
__global__ void gather_rows_scalar_kernel(DT* __restrict__ dst, long long ld_dst, const DT* __restrict__ src,
                                          long long ld_src, const IdxT* __restrict__ list, long long off,
                                          long long count, int n) {
  const long long total = count * n;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long u = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; u < total; u += stride) {
    const long long r = u / n;
    const int c = static_cast<int>(u - r * n);
    dst[r * ld_dst + c] = *static_cast<const volatile DT*>(src + list_at(list, r, off) * ld_src + c);
  }
}

__device__ __forceinline__ uint4 add16(uint4 a, uint4 b, float) {
  a.x = __float_as_uint(__uint_as_float(a.x) + __uint_as_float(b.x));
  a.y = __float_as_uint(__uint_as_float(a.y) + __uint_as_float(b.y));
  a.z = __float_as_uint(__uint_as_float(a.z) + __uint_as_float(b.z));
  a.w = __float_as_uint(__uint_as_float(a.w) + __uint_as_float(b.w));
  return a;
}
__device__ __forceinline__ uint32_t add_bf16x2(uint32_t a, uint32_t b) {
  const float lo = __uint_as_float(a << 16) + __uint_as_float(b << 16);
  const float hi = __uint_as_float(a & 0xffff0000u) + __uint_as_float(b & 0xffff0000u);
  const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint4 add16(uint4 a, uint4 b, __nv_bfloat16) {
  a.x = add_bf16x2(a.x, b.x);
  a.y = add_bf16x2(a.y, b.y);
  a.z = add_bf16x2(a.z, b.z);
  a.w = add_bf16x2(a.w, b.w);
  return a;
}

// dst[list[i] - off, :] += src[i, :]; the entries of `list` are distinct.
template <typename IdxT, typename DT>
__global__ void __launch_bounds__(kThreads) scatter_add_rows_kernel(
    char* __restrict__ dst, long long dst_stride, const char* __restrict__ src, long long src_stride,
    const IdxT* __restrict__ list, long long off, long long count, int units) {
  const long long total = count * units;
  const long long stride = static_cast<long long>(gridDim.x) * kThreads;
  long long u = static_cast<long long>(blockIdx.x) * kThreads + threadIdx.x;
  for (; u + (kUnroll - 1) * stride < total; u += kUnroll * stride) {
    uint4 v[kUnroll];
    char* d[kUnroll];
#pragma unroll
    for (int k = 0; k < kUnroll; ++k) {
      const long long uu = u + k * stride;
      const long long r = uu / units;
      const int c = static_cast<int>(uu - r * units);
      v[k] = ld_peer16(src + r * src_stride + c * 16);
      d[k] = dst + list_at(list, r, off) * dst_stride + c * 16;
    }
#pragma unroll
    for (int k = 0; k < kUnroll; ++k) {
      uint4* dp = reinterpret_cast<uint4*>(d[k]);
      *dp = add16(*dp, v[k], DT{});
    }
  }
  for (; u < total; u += stride) {
    const long long r = u / units;
    const int c = static_cast<int>(u - r * units);
    uint4* dp = reinterpret_cast<uint4*>(dst + list_at(list, r, off) * dst_stride + c * 16);
    *dp = add16(*dp, ld_peer16(src + r * src_stride + c * 16), DT{});
  }
}

template <typename IdxT, typename DT>
__global__ void scatter_add_rows_scalar_kernel(DT* __restrict__ dst, long long ld_dst, const DT* __restrict__ src,
                                               long long ld_src, const IdxT* __restrict__ list, long long off,
                                               long long count, int n) {
  const long long total = count * n;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long u = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; u < total; u += stride) {
    const long long r = u / n;
    const int c = static_cast<int>(u - r * n);
    DT* dp = dst + list_at(list, r, off) * ld_dst + c;
    *dp = from_float<DT>(to_float(*dp) + to_float(*static_cast<const volatile DT*>(src + r * ld_src + c)));
  }
}

// fp32 accumulator variant: dst is fp32, src rows are bf16 (the peers' partials, each rounded
// once); 16 bytes of src = 8 values = 32 bytes of dst.  Keeps a sum over many ranks from being
// rounded to bf16 after every addend.
template <typename IdxT>
__global__ void __launch_bounds__(kThreads) scatter_add_rows_bf16_to_f32_kernel(
    float* __restrict__ dst, long long ld_dst, const char* __restrict__ src, long long src_stride,
    const IdxT* __restrict__ list, long long off, long long count, int units) {
  const long long total = count * units;
  const long long stride = static_cast<long long>(gridDim.x) * kThreads;
  for (long long u = static_cast<long long>(blockIdx.x) * kThreads + threadIdx.x; u < total; u += stride) {
    const long long r = u / units;
    const int c = static_cast<int>(u - r * units);
    const uint4 v = ld_peer16(src + r * src_stride + c * 16);
    float4* dp = reinterpret_cast<float4*>(dst + list_at(list, r, off) * ld_dst + c * 8);
    float4 a = dp[0], b = dp[1];
    a.x += __uint_as_float(v.x << 16); a.y += __uint_as_float(v.x & 0xffff0000u);
    a.z += __uint_as_float(v.y << 16); a.w += __uint_as_float(v.y & 0xffff0000u);
    b.x += __uint_as_float(v.z << 16); b.y += __uint_as_float(v.z & 0xffff0000u);
    b.z += __uint_as_float(v.w << 16); b.w += __uint_as_float(v.w & 0xffff0000u);
    dp[0] = a;
    dp[1] = b;
  }
}

template <typename IdxT>
__global__ void scatter_add_rows_bf16_to_f32_scalar_kernel(float* __restrict__ dst, long long ld_dst,
                                                           const __nv_bfloat16* __restrict__ src, long long ld_src,
                                                           const IdxT* __restrict__ list, long long off,
                                                           long long count, int n) {
  const long long total = count * n;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long u = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; u < total; u += stride) {
    const long long r = u / n;
    const int c = static_cast<int>(u - r * n);
    dst[list_at(list, r, off) * ld_dst + c] += to_float(*static_cast<const volatile __nv_bfloat16*>(src + r * ld_src + c));
  }
}

// ---------------------------------------------------------------------------------------------
// Flag-synchronised multi-peer kernels: ONE launch pulls from (or combines the partials of) every
// peer, and the inter-rank ordering lives inside the kernel — each source segment is guarded by an
// epoch flag its owner writes into THIS rank's signal pad (st.release.sys over NVLink) after its
// data is complete; a block spins (ld.acquire.sys + nanosleep) on the flag of the segment it is
// about to read.  No host barrier, no collective, no per-peer launch: at 8 ranks a forward is
// publish + signal + pull + two products, whatever the number of peers.  Buffers are double
// buffered by epoch parity by the caller, so no "done reading" handshake is needed (dist.py).
// One rank per GPU only: kernels of different ranks wait on one another (B200_PROFILING.md).

struct PullSeg {
  const char* src;          // peer buffer (row 0 of the peer's published shard)
  const void* list;         // rows wanted from it (device, IdxT), relative to `src`
  const unsigned long long* flag;   // this rank's pad slot the owner of `src` writes its epoch to
  long long count;          // rows
  long long dst_row;        // first destination row of the segment
};
constexpr int kMaxSegs = 16;
struct PullArgs {
  PullSeg seg[kMaxSegs];
  int nseg;
};

__device__ __forceinline__ void wait_flag(const unsigned long long* flag, unsigned long long epoch) {
  if (threadIdx.x == 0) {
    unsigned long long v;
    for (;;) {
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
      if (v >= epoch) break;
      __nanosleep(200);
    }
  }
  __syncthreads();
}

constexpr int kPullThreads = 128;   // fits the CTA slot the overlapped product leaves free per SM

// TMA pull: one warp per CTA drives a ring of kStages shared-memory stages.  Every wanted row is one
// cp.async.bulk (global -> shared) straight from the owner's HBM over NVLink, completion counted on
// the stage's mbarrier; a landed stage leaves as ONE bulk store (shared -> global; destination rows
// are consecutive).  The loads of the next kAhead batches are in flight while a batch is waited
// for: 3 x 16 KB per CTA, ~7 MB chip-wide — the bytes in flight NVLink's ~3 us round trip needs at
// 700+ GB/s — for 32 threads and a handful of registers per SM, so the product it overlaps keeps
// its occupancy.  Stage reuse: load #i refills the stage of load #i-kStages, whose store is at
// least two commits old when at most kAhead = kStages-2 loads run ahead; waiting until at most one
// store group is pending therefore guarantees that store has finished reading the stage.
constexpr int kStages = 5;
constexpr int kAhead = kStages - 2;
constexpr int kStageBytes = 16 * 1024;

__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

template <typename IdxT>
__global__ void __launch_bounds__(32) pull_rows_tma_kernel(char* __restrict__ dst, long long dst_stride, long long src_stride,
                                                          const PullArgs a, unsigned long long epoch, uint32_t row_bytes) {
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  const int lane = threadIdx.x;
  const int rows_per_stage = kStageBytes / row_bytes;
  if (lane == 0)
    for (int i = 0; i < kStages; ++i) mbar_init(&bars[i], 1);
  fence_mbar_init();
  __syncwarp();
  const uint64_t pol = l2_policy_evict_first();
  uint32_t phase_bits = 0;     // bit i = parity to wait for on stage i
  long long issued = 0, done = 0;   // batches this CTA has issued / retired, over all segments (ring position)
  for (int s = 0; s < a.nseg; ++s) {
    const PullSeg sg = a.seg[s];
    if (sg.count == 0) continue;
    if (lane == 0) {
      unsigned long long v;
      for (;;) {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(sg.flag) : "memory");
        if (v >= epoch) break;
        __nanosleep(200);
      }
    }
    __syncwarp();
    const IdxT* list = static_cast<const IdxT*>(sg.list);
    const long long nb = (sg.count + rows_per_stage - 1) / rows_per_stage;      // batches of the segment
    const long long mine = blockIdx.x < nb ? (nb - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    auto issue = [&](long long k) {   // k-th batch of this CTA in this segment
      const long long batch = blockIdx.x + k * gridDim.x;
      const int st = static_cast<int>(issued % kStages);
      const long long r0 = batch * rows_per_stage;
      const int cnt = static_cast<int>(sg.count - r0 < rows_per_stage ? sg.count - r0 : rows_per_stage);
      if (issued >= kStages) {       // the store that last used this stage must have finished reading it
        if (lane == 0) bulk_wait_read<1>();
        __syncwarp();
      }
      if (lane == 0) mbar_arrive_expect_tx(&bars[st], static_cast<uint32_t>(cnt) * row_bytes);
      __syncwarp();
      for (int r = lane; r < cnt; r += 32)
        tma_bulk_g2s(smem + st * kStageBytes + r * row_bytes, sg.src + static_cast<long long>(list[r0 + r]) * src_stride, row_bytes,
                     &bars[st], pol);
      ++issued;
    };
    long long k_issue = 0;
    for (; k_issue < mine && k_issue < kAhead; ++k_issue) issue(k_issue);
    for (long long k = 0; k < mine; ++k) {
      if (k_issue < mine) issue(k_issue++);
      const int st = static_cast<int>(done % kStages);
      mbar_wait(&bars[st], (phase_bits >> st) & 1u);
      phase_bits ^= 1u << st;
      const long long batch = blockIdx.x + k * gridDim.x;
      const long long r0 = batch * rows_per_stage;
      const int cnt = static_cast<int>(sg.count - r0 < rows_per_stage ? sg.count - r0 : rows_per_stage);
      if (lane == 0) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        bulk_s2g(dst + (sg.dst_row + r0) * dst_stride, smem + st * kStageBytes, static_cast<uint32_t>(cnt) * row_bytes);
        bulk_commit();
      }
      __syncwarp();
      ++done;
    }
  }
  if (lane == 0) bulk_wait_read<0>();
  __syncwarp();
}

// Register fallback (rows that are not packed / too wide for a stage): 16-byte loads, kUnroll in flight.
template <typename IdxT>
__global__ void __launch_bounds__(kPullThreads) pull_rows_multi_kernel(char* __restrict__ dst, long long dst_stride,
                                                                      long long src_stride, const PullArgs a,
                                                                      unsigned long long epoch, int units) {
  for (int s = 0; s < a.nseg; ++s) {
    const PullSeg sg = a.seg[s];
    if (sg.count == 0) continue;
    wait_flag(sg.flag, epoch);
    const IdxT* list = static_cast<const IdxT*>(sg.list);
    const long long total = sg.count * units;
    const long long stride = static_cast<long long>(gridDim.x) * kPullThreads;
    long long u = static_cast<long long>(blockIdx.x) * kPullThreads + threadIdx.x;
    for (; u + (kUnroll - 1) * stride < total; u += kUnroll * stride) {
      uint4 v[kUnroll];
      long long drow[kUnroll];
      int c[kUnroll];
#pragma unroll
      for (int k = 0; k < kUnroll; ++k) {
        const long long uu = u + k * stride;
        drow[k] = uu / units;
        c[k] = static_cast<int>(uu - drow[k] * units);
        v[k] = ld_peer16(sg.src + static_cast<long long>(list[drow[k]]) * src_stride + c[k] * 16);
      }
#pragma unroll
      for (int k = 0; k < kUnroll; ++k)
        *reinterpret_cast<uint4*>(dst + (sg.dst_row + drow[k]) * dst_stride + c[k] * 16) = v[k];
    }
    for (; u < total; u += stride) {
      const long long r = u / units;
      const int c = static_cast<int>(u - r * units);
      *reinterpret_cast<uint4*>(dst + (sg.dst_row + r) * dst_stride + c * 16) =
          ld_peer16(sg.src + static_cast<long long>(list[r]) * src_stride + c * 16);
    }
  }
}

struct CombineSeg {
  const char* src;          // peer partial rows for this rank's shard (first row of the segment)
  const int* inv;           // this rank's rows -> index into the segment, or -1 (device, int32[rows])
  const unsigned long long* flag;
};
struct CombineArgs {
  CombineSeg seg[kMaxSegs];
  int nseg;
};

// acc[row, :] += sum over peers (in the order of `a.seg`, i.e. ascending rank: a fixed summation
// order) of the peer's partial row, for the rows the peer holds.  One 16-byte unit of the source
// dtype per thread; AccT = float for bf16 sources (rounded once by the caller), = source for fp32.
template <typename SrcT>
__device__ __forceinline__ void add_unit(float* d, const uint4& v) {
  if constexpr (sizeof(SrcT) == 4) {
    float4 x = *reinterpret_cast<float4*>(d);
    x.x += __uint_as_float(v.x); x.y += __uint_as_float(v.y); x.z += __uint_as_float(v.z); x.w += __uint_as_float(v.w);
    *reinterpret_cast<float4*>(d) = x;
  } else {
    float4 x = reinterpret_cast<float4*>(d)[0], y = reinterpret_cast<float4*>(d)[1];
    x.x += __uint_as_float(v.x << 16); x.y += __uint_as_float(v.x & 0xffff0000u);
    x.z += __uint_as_float(v.y << 16); x.w += __uint_as_float(v.y & 0xffff0000u);
    y.x += __uint_as_float(v.z << 16); y.y += __uint_as_float(v.z & 0xffff0000u);
    y.z += __uint_as_float(v.w << 16); y.w += __uint_as_float(v.w & 0xffff0000u);
    reinterpret_cast<float4*>(d)[0] = x;
    reinterpret_cast<float4*>(d)[1] = y;
  }
}

// The unit -> thread mapping is the same for every segment, so one thread adds all peers'
// contributions to its units, in segment order; kUnroll peer loads in flight per thread.
template <typename SrcT>
__global__ void __launch_bounds__(kPullThreads) combine_rows_multi_kernel(float* __restrict__ acc, long long ld_acc,
                                                                         long long src_stride, const CombineArgs a,
                                                                         unsigned long long epoch, long long rows, int units) {
  constexpr int kPer = 16 / sizeof(SrcT);   // values per 16-byte unit: 4 fp32 or 8 bf16
  const long long total = rows * units;
  const long long stride = static_cast<long long>(gridDim.x) * kPullThreads;
  for (int s = 0; s < a.nseg; ++s) {
    const CombineSeg sg = a.seg[s];
    wait_flag(sg.flag, epoch);
    for (long long u0 = static_cast<long long>(blockIdx.x) * kPullThreads + threadIdx.x; u0 < total; u0 += kUnroll * stride) {
      uint4 v[kUnroll];
      float* d[kUnroll];
#pragma unroll
      for (int k = 0; k < kUnroll; ++k) {
        const long long u = u0 + k * stride;
        d[k] = nullptr;
        if (u < total) {
          const long long r = u / units;
          const int j = sg.inv[r];
          if (j >= 0) {
            const int c = static_cast<int>(u - r * units);
            v[k] = ld_peer16(sg.src + static_cast<long long>(j) * src_stride + c * 16);
            d[k] = acc + r * ld_acc + c * kPer;
          }
        }
      }
#pragma unroll
      for (int k = 0; k < kUnroll; ++k)
        if (d[k] != nullptr) add_unit<SrcT>(d[k], v[k]);
    }
    __syncthreads();
  }
}

struct SignalArgs {
  unsigned long long* slot[kMaxSegs];   // per peer: where this rank's epoch goes in the peer's pad
  int n;
};
// After everything earlier on the stream (the publish of this rank's data): tell every peer.
__global__ void signal_peers_kernel(const SignalArgs a, unsigned long long epoch) {
  __threadfence_system();
  const int i = threadIdx.x;
  if (i < a.n) asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(a.slot[i]), "l"(epoch) : "memory");
}

template <typename IdxT, typename ValT>
__global__ void gather_vals_kernel(const ValT* __restrict__ val, const IdxT* __restrict__ perm, long long nnz,
                                   ValT* __restrict__ out) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; q < nnz; q += stride)
    out[q] = val[perm[q]];
}

template <typename IdxT, typename DT>
int rows_impl(bool add, void* dst, int64_t ld_dst, const void* src, int64_t ld_src, const void* list,
              int64_t off, int64_t count, int64_t n, int max_ctas, cudaStream_t stream) {
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  const bool vec = (n * sizeof(DT)) % 16 == 0 && (ld_dst * sizeof(DT)) % 16 == 0 && (ld_src * sizeof(DT)) % 16 == 0 &&
                   ((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 15) == 0;
  const IdxT* l = static_cast<const IdxT*>(list);
  if (vec) {
    const int units = static_cast<int>(n * sizeof(DT) / 16);
    const int grid = grid_for((count * units + kUnroll - 1) / kUnroll, kThreads, max_ctas, dev.sms);
    if (add)
      scatter_add_rows_kernel<IdxT, DT><<<grid, kThreads, 0, stream>>>(
          static_cast<char*>(dst), ld_dst * sizeof(DT), static_cast<const char*>(src), ld_src * sizeof(DT), l, off, count, units);
    else
      gather_rows_kernel<IdxT><<<grid, kThreads, 0, stream>>>(
          static_cast<char*>(dst), ld_dst * sizeof(DT), static_cast<const char*>(src), ld_src * sizeof(DT), l, off, count, units);
  } else {
    const int grid = grid_for(count * n, 256, max_ctas, dev.sms);
    if (add)
      scatter_add_rows_scalar_kernel<IdxT, DT><<<grid, 256, 0, stream>>>(
          static_cast<DT*>(dst), ld_dst, static_cast<const DT*>(src), ld_src, l, off, count, static_cast<int>(n));
    else
      gather_rows_scalar_kernel<IdxT, DT><<<grid, 256, 0, stream>>>(
          static_cast<DT*>(dst), ld_dst, static_cast<const DT*>(src), ld_src, l, off, count, static_cast<int>(n));
  }
  return launched();
}

int rows_dispatch(bool add, void* dst, int64_t ld_dst, const void* src, int64_t ld_src, const void* list,
                  int idx_dtype, int64_t off, int64_t count, int64_t n, int dense_dtype, int max_ctas,
                  cudaStream_t stream) {
  if (count == 0 || n == 0) return OFSPMM_OK;
  return dispatch_dense(dense_dtype, [&](auto dense) {
    return dispatch_idx(idx_dtype, [&](auto idx) {
      return rows_impl<typename decltype(idx)::type, typename decltype(dense)::type>(add, dst, ld_dst, src, ld_src, list,
                                                                                    off, count, n, max_ctas, stream);
    });
  });
}

}  // namespace

int launch_gather_rows(void* dst, int64_t ld_dst, const void* src, int64_t ld_src, const void* list,
                       int idx_dtype, int64_t idx_offset, int64_t count, int64_t n, int dense_dtype,
                       int max_ctas, cudaStream_t stream) {
  return rows_dispatch(false, dst, ld_dst, src, ld_src, list, idx_dtype, idx_offset, count, n, dense_dtype, max_ctas, stream);
}

int launch_scatter_add_rows(void* dst, int64_t ld_dst, const void* src, int64_t ld_src, const void* list,
                            int idx_dtype, int64_t idx_offset, int64_t count, int64_t n, int dense_dtype,
                            int max_ctas, cudaStream_t stream) {
  return rows_dispatch(true, dst, ld_dst, src, ld_src, list, idx_dtype, idx_offset, count, n, dense_dtype, max_ctas, stream);
}

int launch_scatter_add_rows_f32(float* dst, int64_t ld_dst, const void* src, int64_t ld_src, const void* list,
                                int idx_dtype, int64_t idx_offset, int64_t count, int64_t n, int src_dtype,
                                int max_ctas, cudaStream_t stream) {
  if (count == 0 || n == 0) return OFSPMM_OK;
  if (src_dtype == OFSPMM_DTYPE_FLOAT)   // fp32 partials: the plain kernel already accumulates in fp32
    return launch_scatter_add_rows(dst, ld_dst, src, ld_src, list, idx_dtype, idx_offset, count, n, src_dtype, max_ctas, stream);
  if (src_dtype != OFSPMM_DTYPE_BFLOAT16) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  const bool vec = n % 8 == 0 && ld_dst % 8 == 0 && ld_src % 8 == 0 &&
                   ((reinterpret_cast<uintptr_t>(dst) & 31) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
  return dispatch_idx(idx_dtype, [&](auto idx) {
    using IdxT = typename decltype(idx)::type;
    const IdxT* l = static_cast<const IdxT*>(list);
    if (vec) {
      const int units = static_cast<int>(n / 8);
      const int grid = grid_for(count * units, kThreads, max_ctas, dev.sms);
      scatter_add_rows_bf16_to_f32_kernel<IdxT><<<grid, kThreads, 0, stream>>>(
          dst, ld_dst, static_cast<const char*>(src), ld_src * 2, l, idx_offset, count, units);
    } else {
      const int grid = grid_for(count * n, 256, max_ctas, dev.sms);
      scatter_add_rows_bf16_to_f32_scalar_kernel<IdxT><<<grid, 256, 0, stream>>>(
          dst, ld_dst, static_cast<const __nv_bfloat16*>(src), ld_src, l, idx_offset, count, static_cast<int>(n));
    }
    return launched();
  });
}

int launch_cast_from_f32(const float* src, void* dst, int64_t count, int dst_dtype, cudaStream_t stream) {
  if (count == 0) return OFSPMM_OK;
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  const int grid = grid_for(count, 256, dev.sms * 8, dev.sms);
  return dispatch_dense(dst_dtype, [&](auto dt) {
    using DT = typename decltype(dt)::type;
    cast_from_f32_kernel<DT><<<grid, 256, 0, stream>>>(src, static_cast<DT*>(dst), count);
    return launched();
  });
}

int launch_signal_peers(void* const* slots, int n, unsigned long long epoch, cudaStream_t stream) {
  if (n < 0 || n > kMaxSegs) return OFSPMM_ERR_INVALID_ARG;
  if (n == 0) return OFSPMM_OK;
  SignalArgs a;
  a.n = n;
  for (int i = 0; i < n; ++i) a.slot[i] = static_cast<unsigned long long*>(slots[i]);
  signal_peers_kernel<<<1, 32, 0, stream>>>(a, epoch);
  return launched();
}

int launch_pull_rows_multi(void* dst, int64_t ld_dst, int64_t ld_src, const ofspmm_pull_seg* segs, int nseg,
                           unsigned long long epoch, int64_t n, int dense_dtype, int idx_dtype, int max_ctas,
                           cudaStream_t stream) {
  if (nseg < 0 || nseg > kMaxSegs) return OFSPMM_ERR_INVALID_ARG;
  const size_t es = dense_dtype == OFSPMM_DTYPE_FLOAT ? 4 : 2;
  if (dense_dtype != OFSPMM_DTYPE_FLOAT && dense_dtype != OFSPMM_DTYPE_BFLOAT16) return OFSPMM_ERR_UNSUPPORTED_DTYPE;
  if ((n * es) % 16 != 0 || (ld_dst * es) % 16 != 0 || (ld_src * es) % 16 != 0 || (reinterpret_cast<uintptr_t>(dst) & 15))
    return OFSPMM_ERR_INVALID_ARG;   // the multi-peer path moves whole 16-byte units
  PullArgs a;
  a.nseg = nseg;
  long long rows = 0;
  for (int i = 0; i < nseg; ++i) {
    if (segs[i].count < 0 || (segs[i].count > 0 && (segs[i].src == nullptr || segs[i].list == nullptr || segs[i].flag == nullptr)))
      return OFSPMM_ERR_INVALID_ARG;
    if (reinterpret_cast<uintptr_t>(segs[i].src) & 15) return OFSPMM_ERR_INVALID_ARG;
    a.seg[i].src = static_cast<const char*>(segs[i].src);
    a.seg[i].list = segs[i].list;
    a.seg[i].flag = static_cast<const unsigned long long*>(segs[i].flag);
    a.seg[i].count = segs[i].count;
    a.seg[i].dst_row = segs[i].dst_row;
    rows += segs[i].count;
  }
  if (rows == 0 || n == 0) return OFSPMM_OK;
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  const int units = static_cast<int>(n * es / 16);
  const size_t row_bytes = static_cast<size_t>(n) * es;
  return dispatch_idx(idx_dtype, [&](auto idx) -> int {
    using IdxT = typename decltype(idx)::type;
    if (ld_dst == n && row_bytes <= static_cast<size_t>(kStageBytes)) {
      // TMA path: destination rows packed (one bulk store per stage), a row fits a stage
      const int rows_per_stage = static_cast<int>(kStageBytes / row_bytes);
      const size_t smem = static_cast<size_t>(kStages) * kStageBytes + kStages * sizeof(uint64_t);
      int grid = max_ctas > 0 ? max_ctas : dev.sms * 2;
      const long long need = (rows + rows_per_stage - 1) / rows_per_stage;
      if (grid > need) grid = static_cast<int>(need < 1 ? 1 : need);
      static KernelLaunchCache cache;  // one per index type
      if (cache.get(dev.ordinal) == 0) {
        OFSPMM_CUDA_OK(cudaFuncSetAttribute(pull_rows_tma_kernel<IdxT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            static_cast<int>(smem)));
        cache.set(dev.ordinal, 1);
      }
      pull_rows_tma_kernel<IdxT><<<grid, 32, smem, stream>>>(static_cast<char*>(dst), ld_dst * es, ld_src * es, a, epoch,
                                                            static_cast<uint32_t>(row_bytes));
    } else {
      int grid = max_ctas > 0 ? max_ctas : dev.sms * 2;
      const long long need = (rows * units + kPullThreads * kUnroll - 1) / (kPullThreads * kUnroll);
      if (grid > need) grid = static_cast<int>(need < 1 ? 1 : need);
      pull_rows_multi_kernel<IdxT><<<grid, kPullThreads, 0, stream>>>(static_cast<char*>(dst), ld_dst * es, ld_src * es, a,
                                                                     epoch, units);
    }
    return launched();
  });
}

int launch_combine_rows_multi(float* acc, int64_t ld_acc, int64_t ld_src, const ofspmm_combine_seg* segs, int nseg,
                              unsigned long long epoch, int64_t rows, int64_t n, int src_dtype, int max_ctas,
                              cudaStream_t stream) {
  if (nseg < 0 || nseg > kMaxSegs) return OFSPMM_ERR_INVALID_ARG;
  return dispatch_dense(src_dtype, [&](auto st) -> int {
    using SrcT = typename decltype(st)::type;
    constexpr size_t es = sizeof(SrcT);
    // one 16-byte source unit = 4 fp32 (16 B of fp32 accumulator) or 8 bf16 (32 B of accumulator)
    constexpr size_t acc_unit = 16 / es * sizeof(float);
    if ((n * es) % 16 != 0 || (ld_src * es) % 16 != 0 || (ld_acc * 4) % acc_unit != 0 ||
        (reinterpret_cast<uintptr_t>(acc) & (acc_unit - 1)))
      return OFSPMM_ERR_INVALID_ARG;
    if (nseg == 0 || rows == 0 || n == 0) return OFSPMM_OK;
    CombineArgs a;
    a.nseg = nseg;
    for (int i = 0; i < nseg; ++i) {
      if (segs[i].src == nullptr || segs[i].inv == nullptr || segs[i].flag == nullptr) return OFSPMM_ERR_INVALID_ARG;
      a.seg[i].src = static_cast<const char*>(segs[i].src);
      a.seg[i].inv = static_cast<const int*>(segs[i].inv);
      a.seg[i].flag = static_cast<const unsigned long long*>(segs[i].flag);
    }
    DevInfo dev;
    if (int rc = get_dev_info(&dev)) return rc;
    const int units = static_cast<int>(n * es / 16);
    int grid = max_ctas > 0 ? max_ctas : dev.sms * 8;
    const long long need = (rows * units + kPullThreads * kUnroll - 1) / (kPullThreads * kUnroll);
    if (grid > need) grid = static_cast<int>(need < 1 ? 1 : need);
    combine_rows_multi_kernel<SrcT><<<grid, kPullThreads, 0, stream>>>(acc, ld_acc, ld_src * es, a, epoch, rows, units);
    return launched();
  });
}

int launch_gather_vals(const void* val, int val_dtype, const void* perm, int idx_dtype, int64_t nnz,
                       void* out, cudaStream_t stream) {
  if (nnz == 0) return OFSPMM_OK;
  DevInfo dev;
  if (int rc = get_dev_info(&dev)) return rc;
  const int grid = grid_for(nnz, 256, dev.sms * 8, dev.sms);
  return dispatch_dense(val_dtype, [&](auto vt) {
    return dispatch_idx(idx_dtype, [&](auto idx) {
      using ValT = typename decltype(vt)::type;
      using IdxT = typename decltype(idx)::type;
      gather_vals_kernel<IdxT, ValT><<<grid, 256, 0, stream>>>(static_cast<const ValT*>(val), static_cast<const IdxT*>(perm),
                                                              nnz, static_cast<ValT*>(out));
      return launched();
    });
  });
}

}  // namespace ofspmm
