// sddmm_bwd_kernels.cuh — SDDMM value gradient and the atomic A^T·dY scatter, both on the same
// merge-path task list and TMA staging as the forward kernel (see spmm_kernels.cuh).
#pragma once
#include "spmm_kernels.cuh"

namespace ofspmm {

struct SddmmParams {
  const void* crow;
  const void* col;
  const void* dY;   // rows x n
  const void* B;    // cols x n
  void* dval;       // nnz
  const void* part;  // int2 or longlong2 entries (PartOf in spmm_kernels.cuh)
  unsigned int* counter;  // dynamic task order (see spmm_merge_kernel); nullptr = static
  long long cols;
  int rows;
  int reserved = 0;  // not read; keeps the parameter layout the narrow kernels were tuned with
  int n;
  int P;
};

// Lanes of one group (LPR consecutive lanes).
template <int LPR>
__device__ __forceinline__ unsigned group_mask(int grp) {
  if constexpr (LPR == 32) return 0xffffffffu;
  return ((1u << LPR) - 1u) << (grp * LPR);
}

// Coalesced write-back of the SDDMM results of non-zeros ns .. ns+cnt_nz-1, staged in sout;
// out-of-range columns (badmask, one bit per staged non-zero and lane) give 0.
template <typename ValT, typename NzT>
__device__ __forceinline__ void store_dval(ValT* dval, NzT ns, const float* sout, int cnt_nz, unsigned badmask, int lane) {
  __syncwarp();
  for (int q0 = 0; q0 < cnt_nz; q0 += 32) {
    const unsigned bad = __shfl_sync(0xffffffffu, badmask, q0 >> 5);
    const int q = q0 + lane;
    if (q < cnt_nz) dval[ns + q] = from_float<ValT>(((bad >> lane) & 1u) ? 0.f : sout[q]);
  }
}

// dval[p] = <dY[i,:], B[col[p],:]>.
// LPR lanes span one dense row (CH chunks of VEC each); the dY row chunk stays in registers while
// the task walks the row's non-zeros.  Hot loop per 4 non-zeros and lane group: one LDS.128 of 4
// column indices, 4·CH coalesced 16-byte gathers in flight, 4 partial dots, then a
// transpose-reduce across the LPR lanes (log2(LPR)+1 shuffles for the 4 results instead of
// 4·log2(LPR)).  Results are staged in shared memory (the stage's unused value array) and written
// back coalesced; out-of-range columns produce 0 (the oracle's convention).
template <typename DT, typename ValT, typename IdxT, int VEC, int LPR, int CH, bool kFull, int ITEMS, int WARPS, typename PartT>
__global__ void __launch_bounds__(WARPS * 32, min_ctas_per_sm<DT, CH>())
sddmm_merge_kernel(const SddmmParams p) {
  using NzT = typename PartOf<PartT>::Nz;
  const PartT* part = static_cast<const PartT*>(p.part);
  constexpr int G = 32 / LPR;
  constexpr bool kVecIdx = sizeof(IdxT) == 4;
  constexpr uint32_t kChunkBytes = LPR * VEC * sizeof(DT);
  using Stage = TaskStage<IdxT, float, ITEMS>;  // .val doubles as the fp32 result staging buffer
  using RV = RowVec<DT, VEC>;
  static_assert(LPR >= 4, "transpose-reduce needs at least 4 lanes per row");

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int grp = lane / LPR;
  const int lig = lane % LPR;
  const unsigned gmask = group_mask<LPR>(grp);
  uint64_t* bar;
  Stage& st = warp_stage<Stage, WARPS>(warp, lane, bar);
  const uint32_t col_sa = smem_u32(st.col);

  const uint64_t pol_stream = l2_policy_evict_first();
  const IdxT* __restrict__ crow = static_cast<const IdxT*>(p.crow);
  const IdxT* __restrict__ col = static_cast<const IdxT*>(p.col);
  ValT* __restrict__ dval = static_cast<ValT*>(p.dval);
  const int n = p.n;
  const uint32_t row_bytes = static_cast<uint32_t>(n) * sizeof(DT);

  // this lane's columns; masked chunks point at column 0 with a zero dY chunk
  const int col0 = lig * VEC;
  uint32_t choff[CH];
  bool chok[CH];
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) {
    chok[ch] = kFull || (col0 + ch * LPR * VEC < n);
    choff[ch] = chok[ch] ? static_cast<uint32_t>(col0 + ch * LPR * VEC) * sizeof(DT) : 0u;
  }
  unsigned long long bl_bits = reinterpret_cast<unsigned long long>(p.B) + (kFull ? choff[0] : 0u);
  asm volatile("" : "+l"(bl_bits));  // one 64-bit register: gather address = IMAD.WIDE.U32
  const char* __restrict__ Bl = reinterpret_cast<const char*>(bl_bits);
  const char* __restrict__ Yl = static_cast<const char*>(p.dY);

  const int total_warps = gridDim.x * WARPS;
  uint32_t phase = 0;
  unsigned pending = 0;

  // task order: static interleave, or drawn from a counter in launch order; two tasks in hand, the
  // next draw in flight during the task, the next partition entry prefetched (spmm_merge_kernel)
  const bool dynamic = p.counter != nullptr;
  auto draw_now = [&]() -> int {
    unsigned drawn = 0;
    if (lane == 0) drawn = atomicAdd(p.counter, 1u);
    return static_cast<int>(__shfl_sync(0xffffffffu, drawn, 0));
  };
  int k = dynamic ? draw_now() : blockIdx.x * WARPS + warp;
  int k1 = dynamic ? draw_now() : k + total_warps;
  for (; k < p.P; k = k1, k1 = dynamic ? static_cast<int>(__shfl_sync(0xffffffffu, pending, 0)) : k1 + total_warps) {
    pending = 0;
    if (dynamic && lane == 0) pending = atomicAdd(p.counter, 1u);
    if (k1 < p.P && lane == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(&part[k1]));
    const PartT ps = PartOf<PartT>::load(&part[k]);
    const PartT pe = PartOf<PartT>::load(&part[k + 1]);
    const int rs = static_cast<int>(ps.x), re = static_cast<int>(pe.x);
    const NzT ns = ps.y;
    const int cnt_nz = static_cast<int>(pe.y - ns);
    if (cnt_nz == 0) continue;
    const StagedTask<IdxT, float> tk = stage_task<false>(st, bar, phase, crow, col, static_cast<const float*>(nullptr),
                                                        rs, ns, re - rs + 1, cnt_nz, p.cols, lane, pol_stream);
    float* sout = st.val;  // sout[e] = result of non-zero ns + e

    int e = 0;
    for (int r = rs; r <= re; ++r) {
      const int e_end = r < re ? task_rel(tk.srow[r - rs + 1], ns) : cnt_nz;
      if (e_end <= e) continue;
      // dY row chunk → registers
      float y[CH][VEC];
      const char* yrow = Yl + static_cast<unsigned long long>(static_cast<uint32_t>(r)) * row_bytes;
#pragma unroll
      for (int ch = 0; ch < CH; ++ch) {
        if (chok[ch]) {
          RV::load(reinterpret_cast<const DT*>(yrow + choff[ch]), y[ch]);
        } else {
#pragma unroll
          for (int i = 0; i < VEC; ++i) y[ch][i] = 0.f;
        }
      }

      auto dot_one = [&](int elem) {  // full dot of one staged element, result in every group lane
        const IdxT c = tk.scol[elem];
        float d = 0.f;
        if (static_cast<unsigned long long>(c) < static_cast<unsigned long long>(p.cols)) {  // group-uniform
          const char* brow = Bl + row_offset(c, row_bytes);
#pragma unroll
          for (int ch = 0; ch < CH; ++ch)
            d = RV::dot(y[ch], load_b<DT, VEC>(brow + (kFull ? ch * kChunkBytes : choff[ch]), 0), d);
        }
#pragma unroll
        for (int off = LPR / 2; off > 0; off >>= 1) d += __shfl_xor_sync(gmask, d, off);
        if (lig == 0) sout[elem] = d;
      };

      if (kVecIdx && !tk.dirty) {
        // slots s = pre_c + e, read as 16-byte chunks of 4; chunk q of the row goes to group q % G.
        // First / last chunk: slots outside the row are masked (no gather, no result written).
        const int s0 = tk.pre_c + e, s1 = tk.pre_c + e_end;
        const int cbase = s0 & ~3;
        const int nchunks = ((s1 + 3) >> 2) - (s0 >> 2);
        // 4 partial dots -> transpose-reduce over the LPR lanes -> writer lanes store valid slots
        auto reduce_store = [&](float (&d)[4], int sa) {
          constexpr int H = LPR / 2, Q = LPR / 4;
          const bool up = (lig & H) != 0;
          float k0 = up ? d[2] : d[0], k1 = up ? d[3] : d[1];
          const float t0 = up ? d[0] : d[2], t1 = up ? d[1] : d[3];
          k0 += __shfl_xor_sync(gmask, t0, H);
          k1 += __shfl_xor_sync(gmask, t1, H);
          const bool uq = (lig & Q) != 0;
          float kv = uq ? k1 : k0;
          const float tv = uq ? k0 : k1;
          kv += __shfl_xor_sync(gmask, tv, Q);
#pragma unroll
          for (int off = Q / 2; off > 0; off >>= 1) kv += __shfl_xor_sync(gmask, kv, off);
          const int slot = sa + (up ? 2 : 0) + (uq ? 1 : 0);
          if ((lig & (Q - 1)) == 0 && slot >= s0 && slot < s1) sout[slot - tk.pre_c] = kv;
        };
        auto edge_chunk = [&](int q) {
          const int sa = cbase + 4 * q;
          const uint4 cn = lds128(col_sa + static_cast<uint32_t>(sa) * 4u);
          const uint32_t c4[4] = {cn.x, cn.y, cn.z, cn.w};
          float d[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            d[u] = 0.f;
            if (sa + u >= s0 && sa + u < s1) {
              const char* brow = Bl + static_cast<unsigned long long>(c4[u]) * row_bytes;
#pragma unroll
              for (int ch = 0; ch < CH; ++ch)
                d[u] = RV::dot(y[ch], load_b<DT, VEC>(brow + (kFull ? ch * kChunkBytes : choff[ch]), 0), d[u]);
            }
          }
          reduce_store(d, sa);
        };
        if (grp == 0) edge_chunk(0);
        int q = grp == 0 ? G : grp;
        const int qend = nchunks - 1;
        if (q < qend) {
          uint32_t ca = col_sa + static_cast<uint32_t>(cbase + 4 * q) * 4u;
          const uint32_t cend = col_sa + static_cast<uint32_t>(cbase + 4 * qend) * 4u;
          int sa = cbase + 4 * q;
          uint4 cn = lds128(ca);
          do {
            const uint32_t c4[4] = {cn.x, cn.y, cn.z, cn.w};
            typename RV::Raw x[4][CH];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const char* brow = Bl + static_cast<unsigned long long>(c4[u]) * row_bytes;
#pragma unroll
              for (int ch = 0; ch < CH; ++ch)
                x[u][ch] = load_b<DT, VEC>(brow + (kFull ? ch * kChunkBytes : choff[ch]), 0);
            }
            ca += 16u * G;
            if (ca < cend) cn = lds128(ca);
            float d[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              d[u] = 0.f;
#pragma unroll
              for (int ch = 0; ch < CH; ++ch) d[u] = RV::dot(y[ch], x[u][ch], d[u]);
            }
            reduce_store(d, sa);
            sa += 4 * G;
            q += G;
          } while (ca < cend);
        }
        if (nchunks > 1 && q == qend) edge_chunk(qend);
      } else {
        for (int el = e + grp; el < e_end; el += G) dot_one(el);
      }
      e = e_end;
    }
    store_dval(dval, ns, sout, cnt_nz, tk.badmask, lane);
  }
}

// Very wide dense rows (n beyond the register tile): loop over the row in LPR*VEC-column steps,
// re-reading the dY chunk from L1 each time.
template <typename DT, typename ValT, typename IdxT, int VEC, int ITEMS, int WARPS, typename PartT>
__global__ void __launch_bounds__(WARPS * 32) sddmm_wide_kernel(const SddmmParams p) {
  using NzT = typename PartOf<PartT>::Nz;
  const PartT* part = static_cast<const PartT*>(p.part);
  using Stage = TaskStage<IdxT, float, ITEMS>;
  using RV = RowVec<DT, VEC>;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  uint64_t* bar;
  Stage& st = warp_stage<Stage, WARPS>(warp, lane, bar);
  const uint64_t pol_stream = l2_policy_evict_first();
  const IdxT* __restrict__ crow = static_cast<const IdxT*>(p.crow);
  const IdxT* __restrict__ col = static_cast<const IdxT*>(p.col);
  const DT* __restrict__ B = static_cast<const DT*>(p.B);
  const DT* __restrict__ dY = static_cast<const DT*>(p.dY);
  ValT* __restrict__ dval = static_cast<ValT*>(p.dval);
  const int n = p.n;
  const int total_warps = gridDim.x * WARPS;
  uint32_t phase = 0;
  for (int k = blockIdx.x * WARPS + warp; k < p.P; k += total_warps) {
    const PartT ps = PartOf<PartT>::load(&part[k]);
    const PartT pe = PartOf<PartT>::load(&part[k + 1]);
    const int rs = static_cast<int>(ps.x), re = static_cast<int>(pe.x);
    const NzT ns = ps.y;
    const int cnt_nz = static_cast<int>(pe.y - ns);
    if (cnt_nz == 0) continue;
    const StagedTask<IdxT, float> tk = stage_task<false>(st, bar, phase, crow, col, static_cast<const float*>(nullptr),
                                                        rs, ns, re - rs + 1, cnt_nz, p.cols, lane, pol_stream);
    float* sout = st.val;
    int e = 0;
    for (int r = rs; r <= re; ++r) {
      const int e_end = r < re ? task_rel(tk.srow[r - rs + 1], ns) : cnt_nz;
      const DT* yrow = dY + static_cast<size_t>(r) * n;
      for (int q = e; q < e_end; ++q) {
        const IdxT cq = tk.scol[q];
        const bool okq = static_cast<unsigned long long>(cq) < static_cast<unsigned long long>(p.cols);
        const DT* brow = B + static_cast<size_t>(okq ? cq : 0) * n;
        float d = 0.f;
        for (int c0 = lane * VEC; okq && c0 < n; c0 += 32 * VEC) {
          float yy[VEC];
          RV::load(yrow + c0, yy);
          d = RV::dot(yy, RV::load_raw(brow + c0), d);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
        if (lane == 0) sout[q] = d;
      }
      if (e_end > e) e = e_end;
    }
    store_dval(dval, ns, sout, cnt_nz, tk.badmask, lane);
  }
}

struct BwdAtomicParams {
  const void* crow;
  const void* col;
  const void* val;
  const void* dY;  // rows x n
  float* acc;      // cols x n fp32 accumulator (zeroed by the caller)
  const void* part;  // int2 or longlong2 entries (PartOf in spmm_kernels.cuh)
  long long cols;
  int rows;
  int reserved = 0;  // not read; keeps the parameter layout the narrow kernels were tuned with
  int n;
  int P;
};

__device__ __forceinline__ void red_add_f32(float* p, const float (&v)[1]) { atomicAdd(p, v[0]); }
__device__ __forceinline__ void red_add_f32(float* p, const float (&v)[4]) {
  asm volatile("red.relaxed.gpu.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v[0]),
               "f"(v[1]), "f"(v[2]), "f"(v[3])
               : "memory");
}
__device__ __forceinline__ void red_add_f32(float* p, const float (&v)[8]) {
  const float a[4] = {v[0], v[1], v[2], v[3]};
  const float b[4] = {v[4], v[5], v[6], v[7]};
  red_add_f32(p, a);
  red_add_f32(p + 4, b);
}

// acc[col[p], :] += val[p] * dY[i, :] with 16-byte vector reductions (red.global.add.v4.f32).
// Route (2) of ofspmm_bwd_b: needs no transposed copy of A, order-nondeterministic like the
// reference's atomic scatter (oneflow/user/kernels/unsorted_segment_sum_kernel_util.cu:96-117).
template <typename DT, typename ValT, typename IdxT, int VEC, int LPR, int CH, int ITEMS, int WARPS, typename PartT>
__global__ void __launch_bounds__(WARPS * 32) bwd_atomic_kernel(const BwdAtomicParams p) {
  using NzT = typename PartOf<PartT>::Nz;
  const PartT* part = static_cast<const PartT*>(p.part);
  constexpr int G = 32 / LPR;
  using Stage = TaskStage<IdxT, ValT, ITEMS>;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int grp = lane / LPR;
  const int lig = lane % LPR;
  uint64_t* bar;
  Stage& st = warp_stage<Stage, WARPS>(warp, lane, bar);

  const uint64_t pol_stream = l2_policy_evict_first();
  const IdxT* __restrict__ crow = static_cast<const IdxT*>(p.crow);
  const IdxT* __restrict__ col = static_cast<const IdxT*>(p.col);
  const ValT* __restrict__ val = static_cast<const ValT*>(p.val);
  const int n = p.n;
  const int col0 = blockIdx.y * (LPR * VEC * CH) + lig * VEC;
  unsigned chmask = 0;
#pragma unroll
  for (int ch = 0; ch < CH; ++ch)
    if (col0 + ch * LPR * VEC < n) chmask |= 1u << ch;
  const DT* __restrict__ dYl = static_cast<const DT*>(p.dY) + col0;
  float* __restrict__ accl = p.acc + col0;

  const int total_warps = gridDim.x * WARPS;
  uint32_t phase = 0;
  for (int k = blockIdx.x * WARPS + warp; k < p.P; k += total_warps) {
    const PartT ps = PartOf<PartT>::load(&part[k]);
    const PartT pe = PartOf<PartT>::load(&part[k + 1]);
    const int rs = static_cast<int>(ps.x), re = static_cast<int>(pe.x);
    const NzT ns = ps.y;
    const int cnt_nz = static_cast<int>(pe.y - ns);
    if (cnt_nz == 0) continue;
    const StagedTask<IdxT, ValT> tk = stage_task<!kIsUnit<ValT>>(st, bar, phase, crow, col, val, rs, ns, re - rs + 1,
                                                                 cnt_nz, p.cols, lane, pol_stream);
    int e = 0;
    for (int r = rs; r <= re; ++r) {
      const int e_end = r < re ? task_rel(tk.srow[r - rs + 1], ns) : cnt_nz;
      if (e_end <= e) continue;
      float y[CH][VEC];
#pragma unroll
      for (int ch = 0; ch < CH; ++ch)
        if (chmask & (1u << ch)) RowVec<DT, VEC>::load(dYl + static_cast<size_t>(r) * n + ch * LPR * VEC, y[ch]);
      for (int q = e + grp; q < e_end; q += G) {
        const IdxT c = tk.scol[q];
        if (static_cast<unsigned long long>(c) >= static_cast<unsigned long long>(p.cols)) continue;  // skipped
        const float v = val_at(tk.sval, q);
        float* dst = accl + static_cast<size_t>(c) * n;
#pragma unroll
        for (int ch = 0; ch < CH; ++ch)
          if (chmask & (1u << ch)) {
            float t[VEC];
#pragma unroll
            for (int i = 0; i < VEC; ++i) t[i] = v * y[ch][i];
            red_add_f32(dst + ch * LPR * VEC, t);
          }
      }
      e = e_end;
    }
  }
}

// out[i] = DT(acc[i]) — the cast that follows an fp32 accumulation for bf16 outputs
// (reference idiom: oneflow/user/kernels/unsorted_segment_sum_kernel.cpp:162-186).
template <typename DT>
__global__ void cast_from_f32_kernel(const float* __restrict__ in, DT* __restrict__ out, long long count) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += stride)
    out[i] = from_float<DT>(in[i]);
}

}  // namespace ofspmm
