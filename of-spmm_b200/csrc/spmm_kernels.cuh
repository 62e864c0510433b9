// spmm_kernels.cuh — merge-path CSR·dense kernels for sm_100a (forward SpMM; also run on the
// transposed CSR for A^T·dY).
//
// Scheduling (SURVEY.md §8a3/a6): the merged list of (row-end, non-zero) items is cut into tasks
// of ITEMS consecutive items; `part[k]` = (first row, first non-zero) of task k comes from the
// device merge-path partitioner.  One warp executes one task at a time (persistent grid, tasks
// interleaved over warps so that concurrently active rows are neighbours → B-row gathers share
// L2 lines).  A task therefore never holds more than ITEMS non-zeros no matter how skewed the row
// lengths are: hub rows of a power-law graph are spread over many warps and stitched together by
// the deterministic segmented fix-up pass below; short rows are packed many-to-a-task.
//
// Data movement per task: the task's col / val / crow slices are staged into shared memory with
// three 1-D TMA bulk copies (cp.async.bulk + mbarrier complete_tx, L2 evict-first since the CSR
// stream is read exactly once).  A short per-task pass neutralises out-of-range column indices
// in the staged copy, so the hot loop is check-free: per 4 non-zeros it issues one 16-byte LDS
// broadcast of 4 column indices, one of 4 values, four IMAD.WIDE addresses and four coalesced
// 16-byte-per-lane gathers of dense rows (float4 or 8 x bf16) feeding fp32 FMAs.
// LPR lanes cover one dense row (vector-per-row when LPR < 32: 32/LPR groups of non-zeros in
// flight per warp instruction, combined with __shfl_xor at the row end; warp-per-row when
// LPR == 32).  Dense widths beyond one register tile are processed as column panels, panel-major
// in time, so the B panel that is being gathered stays L2-resident.
//
// Output: rows that start and end inside a task are streamed to C once (st.global.cs).  The
// trailing partial row of a task goes to carry[k] (fp32); a row that ends in task k but started
// earlier goes to C (fp32 output) or head[k] (bf16 output, to round only once); fixup_kernel adds
// carries in ascending task order — no atomics, bitwise reproducible.
#pragma once
#include "common.cuh"

#ifndef OFSPMM_B_LOAD
#define OFSPMM_B_LOAD 0  // 0: ld.global.nc   1: + L1::no_allocate   2: 1 + L2 evict_last   3: L1 allocate + L2 evict_last
#endif

namespace ofspmm {

// Resident CTAs per SM the kernels are compiled for (4 warps per CTA): sets the register cap.
// Measured on B200 (tools/sweep_fwd.py, profiles/r1_tuning_sweeps.md): fp32 rows run best at 36
// warps/SM with 54 registers, bf16 rows (8 accumulators + unpacking) at 32 warps/SM with 60.
template <typename DT, int CH>
constexpr int min_ctas_per_sm() {
#ifdef OFSPMM_MIN_CTAS
  return CH == 1 ? OFSPMM_MIN_CTAS : (CH == 2 ? 6 : 4);
#else
  return CH == 1 ? (sizeof(DT) == 4 ? 9 : 8) : (CH == 2 ? 6 : 4);
#endif
}

struct FwdParams {
  const void* crow;
  const void* col;
  const void* val;
  const void* B;
  void* C;
  const void* part;  // P+1 split points (row, nz): int2, or longlong2 for wide matrices (PartOf below)
  float* carry;      // P x n fp32
  float* head;       // P x n fp32 (only for non-fp32 outputs)
  long long cols;    // K
  int rows;          // M
  int reserved = 0;  // not read; keeps the parameter layout the narrow kernels were tuned with
  int n;             // dense width
  int P;             // number of tasks
  int panels;        // column panels of LPR*VEC*CH columns each
  long long ldb;     // row stride of B in elements (>= n)
  long long ldc;     // row stride of C in elements (>= n)
  const void* bias;  // n elements of the dense dtype (kFwdBias)
  unsigned int* counter;  // dynamic task order: zeroed before the launch; nullptr = static
  unsigned flags;    // kFwd* epilogue bits
  int max_tasks;     // tasks a warp runs before its CTA may retire (0: until the list is empty)
  float* acc32;      // rows x n fp32 accumulator of a multi-pass product with a 16-bit output (kFwdAcc32*)
};

// Epilogue bits (= OFSPMM_FWD_* of include/ofspmm.h).  A row's epilogue runs exactly once, where
// its complete fp32 sum is known: in the merge kernel for rows that live inside one task, in the
// fix-up kernel for rows stitched from several tasks.
constexpr unsigned kFwdAccumulate = 1u;  // C += A·B instead of C = A·B
constexpr unsigned kFwdBias = 2u;        // + bias[j]
constexpr unsigned kFwdRelu = 4u;        // max(., 0)
// 16-bit outputs only: a product computed in several accumulate passes (column buckets of the
// multi-GPU path) keeps its running row sums in fp32 between the passes, so the result is rounded
// to bf16 exactly once, like a single-pass product.
constexpr unsigned kFwdAcc32In = 32u;    // add the fp32 row of acc32 to this pass's sum
constexpr unsigned kFwdAcc32Out = 64u;   // store the fp32 sum into acc32 instead of C (no epilogue)
// Mean aggregation: the complete row sum is divided by the row's stored-entry count, first thing in
// the epilogue.  Never combined with kFwdAccumulate / kFwdAcc32* (rejected in api.cu): for fp32
// rows stitched from several tasks the merge kernel folds the old C into the final segment before
// the fix-up adds the carries, so a division in the fix-up would divide the old C as well.
constexpr unsigned kFwdMean = 128u;

// Task partition entry: (first row, first non-zero) of a task.  Matrices with fewer than 2^31-1
// non-zeros use 8-byte int2 entries; wider ones ("wide", int64 indices only) 16-byte longlong2
// entries whose .y is the 64-bit non-zero offset (.x still holds a row < 2^31-1).  Only the task
// start is 64-bit: everything inside a task (e0, e1, cnt_nz, crow[r] - ns) is bounded by ITEMS.
template <typename PartT> struct PartOf;
template <> struct PartOf<int2> {
  using Nz = int;
  __device__ __forceinline__ static int2 load(const int2* p) { return __ldg(p); }
};
template <> struct PartOf<longlong2> {
  using Nz = long long;
  __device__ __forceinline__ static longlong2 load(const longlong2* p) { return __ldg(p); }
};

// Position of a non-zero (a crow value) relative to the task start ns; the result is < ITEMS.
template <typename IdxT, typename NzT>
__device__ __forceinline__ int task_rel(IdxT v, NzT ns) {
  if constexpr (sizeof(NzT) == 4) return static_cast<int>(v) - ns;
  else return static_cast<int>(static_cast<long long>(v) - ns);
}

// 1 / d for a row count d >= 1 without the slow-path subroutine call of the IEEE division (that
// call site costs registers, and spills, in every kernel carrying the epilogue, mean or not):
// reciprocal estimate refined by one Newton step.  The mean is sum * (1/d): within 1.5 ulp of the
// correctly rounded quotient.
__device__ __forceinline__ float recip_count(float d) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
  return fmaf(fmaf(-d, r, 1.f), r, r);
}

// acc (/ len) (+ old C) (+ bias) (relu) for VEC consecutive columns starting at column `c0` of a
// row with `len` stored entries (read only for kFwdMean; an empty row keeps its sum of 0).
template <typename DT, int VEC>
__device__ __forceinline__ void row_epilogue(float (&acc)[VEC], const DT* c_old, const void* bias, int c0,
                                             unsigned flags, bool add_old, float len) {
  if ((flags & kFwdMean) && len > 0.f) {
    const float inv = recip_count(len);
#pragma unroll
    for (int i = 0; i < VEC; ++i) acc[i] *= inv;
  }
  if (add_old) {
    float o[VEC];
    RowVec<DT, VEC>::load(c_old, o);
#pragma unroll
    for (int i = 0; i < VEC; ++i) acc[i] += o[i];
  }
  if (flags & kFwdBias) {
    float b[VEC];
    RowVec<DT, VEC>::load(static_cast<const DT*>(bias) + c0, b);
#pragma unroll
    for (int i = 0; i < VEC; ++i) acc[i] += b[i];
  }
  if (flags & kFwdRelu) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) acc[i] = fmaxf(acc[i], 0.f);
  }
}

template <typename IdxT, typename ValT, int ITEMS>
struct alignas(16) TaskStage {
  static constexpr int kPadI = 2 * (16 / sizeof(IdxT));
  static constexpr int kPadV = 2 * (16 / sizeof(ValT));
  IdxT col[ITEMS + kPadI];
  IdxT crow[ITEMS + 2 * kPadI];
  ValT val[ITEMS + kPadV];
};
// A pattern matrix stages no values.
template <typename IdxT, int ITEMS>
struct alignas(16) TaskStage<IdxT, UnitVal, ITEMS> {
  static constexpr int kPadI = 2 * (16 / sizeof(IdxT));
  IdxT col[ITEMS + kPadI];
  IdxT crow[ITEMS + 2 * kPadI];
};

// Shared-memory address of the staged values (0 for a pattern matrix, which stages none).
template <typename IdxT, typename ValT, int ITEMS>
__device__ __forceinline__ uint32_t staged_val_addr(TaskStage<IdxT, ValT, ITEMS>& st) {
  if constexpr (kIsUnit<ValT>) return 0u;
  else return smem_u32(st.val);
}

// Where element e of a `count`-element global slice starting at `src` lands in the staging array
// (dst[pre + e]) and which part of it is a 16-byte aligned body a TMA bulk copy can move.
template <typename T>
__device__ __forceinline__ void seg_plan(const T* src, int count, int& pre, int& head, int& body) {
  constexpr int EPV = 16 / sizeof(T);
  pre = static_cast<int>((reinterpret_cast<uintptr_t>(src) & 15) / sizeof(T));
  head = (EPV - pre) & (EPV - 1);
  if (head > count) head = count;
  body = ((count - head) / EPV) * EPV;
}

// Ragged ends (< 16 bytes each side) are moved by lanes with ordinary loads.
template <typename T>
__device__ __forceinline__ void seg_copy_edges(T* dst, const T* src, int count, int pre, int head,
                                               int body, int lane) {
  const int edge = count - body;  // head + tail elements, at most 2*(EPV-1)
  if (lane < edge) {
    const int e = lane < head ? lane : body + lane;
    dst[pre + e] = src[e];
  }
}

// One task's CSR slices in shared memory.
template <typename IdxT, typename ValT>
struct StagedTask {
  const IdxT* scol;  // scol[e] = col[ns + e]
  const ValT* sval;  // sval[e] = val[ns + e]   (unused when values are not staged)
  const IdxT* srow;  // srow[i] = crow[rs + i]
  int pre_c, pre_v;  // slot of element 0 inside st.col / st.val (address alignment phase)
  // lane i holds the bit mask of out-of-range elements 32*i .. 32*i+31 of the task
  unsigned badmask;
  // some column index of the task lies outside [0, cols): the task takes the per-element checked
  // path (the staged copy is left untouched, nothing is gathered for such an element)
  bool dirty;
};

// Stages crow[rs..re], col[ns..ne) and (optionally) val[ns..ne) of a task: TMA bulk copies for
// the 16-byte aligned bodies, lanes for the ragged edges, then waits for the bytes to land and
// scans the column indices once: a task whose indices are all inside [0, cols) runs the check-free
// vector loop; a task with an out-of-range index is flagged `dirty` and runs a per-element checked
// loop that issues no load for such an element (so NaN / Inf in unrelated B rows cannot leak in).
template <bool kWithVal, typename IdxT, typename ValT, int ITEMS, typename NzT>
__device__ __forceinline__ StagedTask<IdxT, ValT> stage_task(
    TaskStage<IdxT, ValT, ITEMS>& st, uint64_t* bar, uint32_t& phase, const IdxT* __restrict__ crow,
    const IdxT* __restrict__ col, const ValT* __restrict__ val, int rs, NzT ns, int cnt_row,
    int cnt_nz, long long cols, int lane, uint64_t pol_stream) {
  int pre_c, head_c, body_c, pre_v = 0, head_v = 0, body_v = 0, pre_r, head_r, body_r;
  seg_plan(col + ns, cnt_nz, pre_c, head_c, body_c);
  if constexpr (kWithVal) seg_plan(val + ns, cnt_nz, pre_v, head_v, body_v);
  seg_plan(crow + rs, cnt_row, pre_r, head_r, body_r);
  const uint32_t tx = static_cast<uint32_t>(body_c * sizeof(IdxT) + body_v * sizeof(ValT) +
                                            body_r * sizeof(IdxT));
  __syncwarp();  // every lane is done reading the previous task's stage
  if (lane == 0 && tx != 0) {
    // order this warp's earlier generic-proxy shared-memory stores (ragged edges, SDDMM result
    // staging; made visible to lane 0 by the __syncwarp above) before the async-proxy writes of the
    // bulk copies into the same bytes
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_arrive_expect_tx(bar, tx);
    if (body_c) tma_bulk_g2s(st.col + pre_c + head_c, col + ns + head_c, body_c * sizeof(IdxT), bar, pol_stream);
    if constexpr (kWithVal) {
      if (body_v) tma_bulk_g2s(st.val + pre_v + head_v, val + ns + head_v, body_v * sizeof(ValT), bar, pol_stream);
    }
    if (body_r) tma_bulk_g2s(st.crow + pre_r + head_r, crow + rs + head_r, body_r * sizeof(IdxT), bar, pol_stream);
  }
  seg_copy_edges(st.col, col + ns, cnt_nz, pre_c, head_c, body_c, lane);
  if constexpr (kWithVal) seg_copy_edges(st.val, val + ns, cnt_nz, pre_v, head_v, body_v, lane);
  seg_copy_edges(st.crow, crow + rs, cnt_row, pre_r, head_r, body_r, lane);
  if (tx != 0) {
    mbar_wait(bar, phase);
    phase ^= 1;
  }
  __syncwarp();
  // indices outside [0, cols) contribute nothing (reference: segment-sum skips them)
  unsigned badmask = 0;
  bool dirty = false;
  for (int e0 = 0; e0 < cnt_nz; e0 += 32) {
    const int e = e0 + lane;
    bool bad = false;
    if (e < cnt_nz) {
      const IdxT c = st.col[pre_c + e];
      bad = static_cast<unsigned long long>(c) >= static_cast<unsigned long long>(cols);
    }
    const unsigned m = __ballot_sync(0xffffffffu, bad);
    if (lane == (e0 >> 5)) badmask = m;
    dirty |= m != 0;
  }
  StagedTask<IdxT, ValT> t;
  t.badmask = badmask;
  t.dirty = dirty;
  t.scol = st.col + pre_c;
  if constexpr (kIsUnit<ValT>) t.sval = nullptr;
  else t.sval = st.val + pre_v;
  t.srow = st.crow + pre_r;
  t.pre_c = pre_c;
  t.pre_v = pre_v;
  return t;
}

// Dense-row gather (16 bytes per lane when vectorised) with the configured cache policy; the raw
// bits stay in registers until the FMAs consume them (bf16 is widened at use, not at load).
template <typename DT, int VEC>
__device__ __forceinline__ typename RowVec<DT, VEC>::Raw load_b(const char* p, uint64_t pol) {
#if OFSPMM_B_LOAD == 0
  (void)pol;
  return RowVec<DT, VEC>::load_raw(reinterpret_cast<const DT*>(p));
#else
  if constexpr (VEC * sizeof(DT) == 16) {
    uint4 w;
#if OFSPMM_B_LOAD == 1
    (void)pol;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(w.x), "=r"(w.y), "=r"(w.z), "=r"(w.w) : "l"(p));
#elif OFSPMM_B_LOAD == 3
    asm volatile("ld.global.nc.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(w.x), "=r"(w.y), "=r"(w.z), "=r"(w.w) : "l"(p), "l"(pol));
#else
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(w.x), "=r"(w.y), "=r"(w.z), "=r"(w.w) : "l"(p), "l"(pol));
#endif
    return w;
  } else {
    (void)pol;
    return RowVec<DT, VEC>::load_raw(reinterpret_cast<const DT*>(p));
  }
#endif
}

// Byte offset of dense row c (already validated, non-negative): one IMAD.WIDE.U32 for int32 ids.
template <typename IdxT>
__device__ __forceinline__ unsigned long long row_offset(IdxT c, uint32_t row_bytes) {
  if constexpr (sizeof(IdxT) == 4) {
    return static_cast<unsigned long long>(static_cast<uint32_t>(c)) * row_bytes;
  } else {
    return static_cast<unsigned long long>(c) * row_bytes;
  }
}

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t addr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  return v;
}

// The 4 staged values at shared-memory byte address va as fp32 (a pattern matrix: four 1s).
template <typename ValT>
__device__ __forceinline__ void lds_vals4(uint32_t va, float (&v4)[4]) {
  if constexpr (kIsUnit<ValT>) {
    (void)va;
    v4[0] = v4[1] = v4[2] = v4[3] = 1.f;
  } else if constexpr (sizeof(ValT) == 4) {
    const uint4 w = lds128(va);
    v4[0] = __uint_as_float(w.x); v4[1] = __uint_as_float(w.y);
    v4[2] = __uint_as_float(w.z); v4[3] = __uint_as_float(w.w);
  } else {
    const uint2 w = lds64(va);
    v4[0] = __uint_as_float(w.x << 16); v4[1] = __uint_as_float(w.x & 0xffff0000u);
    v4[2] = __uint_as_float(w.y << 16); v4[3] = __uint_as_float(w.y & 0xffff0000u);
  }
}

// This warp's task stage, and its mbarrier initialised for one arrival, in the dynamic shared memory
// of a merge-path kernel: WARPS stages, then WARPS mbarriers (kMergeSmem in launch.cuh).
template <typename Stage, int WARPS>
__device__ __forceinline__ Stage& warp_stage(int warp, int lane, uint64_t*& bar) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Stage* stages = reinterpret_cast<Stage*>(smem_raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + sizeof(Stage) * WARPS);
  bar = &bars[warp];
  if (lane == 0) mbar_init(bar, 1);
  fence_mbar_init();
  __syncwarp();
  return stages[warp];
}

// kFull: n is a whole number of LPR*VEC*CH-column tiles, so no lane is ever masked and the chunk
// offsets are immediates.  Otherwise masked chunks are pointed at column 0 (a valid address:
// their loads are harmless duplicates) and only the stores are predicated.
template <typename DT, typename ValT, typename IdxT, int VEC, int LPR, int CH, bool kFull, bool kRowPar, int ITEMS, int WARPS,
          typename PartT>
__global__ void __launch_bounds__(WARPS * 32, min_ctas_per_sm<DT, CH>())
spmm_merge_kernel(const FwdParams p) {
  using NzT = typename PartOf<PartT>::Nz;
  constexpr int G = 32 / LPR;  // groups of lanes working on different non-zeros
  constexpr bool kF32Out = sizeof(DT) == 4;
  constexpr bool kVecIdx = sizeof(IdxT) == 4;  // 16-byte LDS path needs 4-byte indices
  constexpr uint32_t kChunkBytes = LPR * VEC * sizeof(DT);
  constexpr bool kUnit = kIsUnit<ValT>;  // pattern matrix: no value stream, every value is 1
  using Stage = TaskStage<IdxT, ValT, ITEMS>;
  using RV = RowVec<DT, VEC>;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int grp = lane / LPR;  // which group of concurrent non-zeros
  const int lig = lane % LPR;  // lane in group -> column chunk
  uint64_t* bar;
  Stage& st = warp_stage<Stage, WARPS>(warp, lane, bar);
  const uint32_t col_sa = smem_u32(st.col);
  const uint32_t val_sa = staged_val_addr(st);

  const uint64_t pol_stream = l2_policy_evict_first();
#if OFSPMM_B_LOAD >= 2
  const uint64_t pol_b = l2_policy_evict_last();
#else
  const uint64_t pol_b = 0;
#endif
  const IdxT* __restrict__ crow = static_cast<const IdxT*>(p.crow);
  const IdxT* __restrict__ col = static_cast<const IdxT*>(p.col);
  const ValT* __restrict__ val = static_cast<const ValT*>(p.val);
  const int n = p.n;
  const uint32_t row_bytes = static_cast<uint32_t>(p.ldb) * sizeof(DT);

  const long long total_tasks = static_cast<long long>(p.P) * p.panels;
  const int total_warps = gridDim.x * WARPS;
  uint32_t phase = 0;

  // Task order.  Static: warp w runs tasks w, w + W, w + 2W, ...  Dynamic (p.counter != nullptr):
  // every task is drawn from a global counter, i.e. handed out in the order warps ask for work, so
  // the rows in flight chip-wide always form ONE contiguous window of the matrix however unevenly
  // the warps progress (keeps the B rows of that window L2-resident — measured -11 % on the
  // Reddit-shaped, -23 % on the products-shaped graph — and evens out the tail).
  // A warp holds two tasks: the one it runs (t) and the next (t1); the draw for the one after is
  // issued at the top of a task and its result is only read at the end (the atomic's latency hides
  // behind the task), and the partition entry of t1 is prefetched into L2 meanwhile.  A warp stops
  // after p.max_tasks tasks (short-lived CTAs for the multi-GPU overlap) and never draws a task it
  // will not run.
  const int total = static_cast<int>(total_tasks);
  const int max_tasks = p.max_tasks > 0 ? p.max_tasks : 0x7fffffff;
  const bool dynamic = p.counter != nullptr;
  auto draw_now = [&]() -> int {
    unsigned drawn = 0;
    if (lane == 0) drawn = atomicAdd(p.counter, 1u);
    return static_cast<int>(__shfl_sync(0xffffffffu, drawn, 0));
  };
  int t = dynamic ? draw_now() : blockIdx.x * WARPS + warp;
  int t1 = dynamic ? (max_tasks > 1 ? draw_now() : total) : t + total_warps;
  for (int done = 0; t < total && done < max_tasks; ++done) {
    unsigned pending = 0;
    const bool more = done + 2 < max_tasks;
    if (dynamic && more && lane == 0) pending = atomicAdd(p.counter, 1u);   // read at the end of the task
    if (t1 < total && lane == 0)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(&static_cast<const PartT*>(p.part)[t1 % p.P]));
    // panel-major: all tasks of column panel 0, then panel 1, ... (keeps the B panel in L2)
    const int panel = t / p.P;
    const int k = t - panel * p.P;
    const int col0 = panel * (LPR * VEC * CH) + lig * VEC;
    unsigned chmask = 0;
    uint32_t choff[CH];  // byte offset of chunk ch from the lane base (0-column for masked chunks)
#pragma unroll
    for (int ch = 0; ch < CH; ++ch) {
      const bool ok = kFull || (col0 + ch * LPR * VEC < n);
      if (ok) chmask |= 1u << ch;
      choff[ch] = ok ? static_cast<uint32_t>(col0 + ch * LPR * VEC) * sizeof(DT) : 0u;
    }
    // lane base: B + first chunk's columns when kFull (other chunks are immediates), else B
    unsigned long long bl_bits = reinterpret_cast<unsigned long long>(p.B) + (kFull ? choff[0] : 0u);
    // opaque to the optimiser: keep base+lane offset as ONE 64-bit register so every gather
    // address is a single IMAD.WIDE.U32 (col * row_bytes + base) instead of IMAD + 64-bit add
    asm volatile("" : "+l"(bl_bits));
    const char* __restrict__ Bl = reinterpret_cast<const char*>(bl_bits);

    const PartT ps = PartOf<PartT>::load(&static_cast<const PartT*>(p.part)[k]);
    const PartT pe = PartOf<PartT>::load(&static_cast<const PartT*>(p.part)[k + 1]);
    const int rs = static_cast<int>(ps.x);
    const NzT ns = ps.y;
    const int re = static_cast<int>(pe.x);
    const NzT ne = pe.y;
    const int cnt_nz = static_cast<int>(ne - ns);
    const StagedTask<IdxT, ValT> tk = stage_task<!kUnit>(st, bar, phase, crow, col, val, rs, ns, re - rs + 1,
                                                         cnt_nz, p.cols, lane, pol_stream);
    // 16-byte LDS path: index chunk and value chunk must share their alignment phase
    const bool vec_ok = kVecIdx && !tk.dirty && (kUnit || (((tk.pre_v - tk.pre_c) & 3) == 0));
    // value byte address of the slot that pairs with index slot 0
    const uint32_t val_s0 = val_sa + static_cast<uint32_t>((tk.pre_v - tk.pre_c) * static_cast<int>(sizeof(ValT)));
    const bool started_earlier = static_cast<NzT>(tk.srow[0]) < ns;

    // nnz-parallel (kRowPar == false): every group walks every row, chunk q of a row goes to group
    // q % G and the groups' partial rows are combined with __shfl_xor at the row end.
    // row-parallel (kRowPar == true, short-row graphs): group g owns rows rs+g, rs+g+G, ... and
    // keeps G independent rows in flight per warp; no cross-group reduction.
    constexpr int kChunkStride = kRowPar ? 1 : G;
    const int chunk_first = kRowPar ? 0 : grp;
    for (int r = kRowPar ? rs + grp : rs; r <= re; r += (kRowPar ? G : 1)) {
      // rows rs..re-1 end in this task; r == re is the trailing partial row (if it has elements)
      // = task_rel(), written out: the int2 instantiations then compile to the code they always had
      const int e0 = r == rs ? 0 : static_cast<int>(static_cast<NzT>(tk.srow[r - rs]) - ns);
      const int e1 = r < re ? static_cast<int>(static_cast<NzT>(tk.srow[r - rs + 1]) - ns) : cnt_nz;
      if (r == re && e1 <= e0) break;

      float acc[CH][VEC];
#pragma unroll
      for (int ch = 0; ch < CH; ++ch)
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[ch][i] = 0.f;

      if (vec_ok) {
        // slots s = pre_c + e.  The row's elements are read as 16-byte chunks of 4 slots; the
        // first / last chunk may contain slots of neighbouring rows (or staging padding), which
        // are masked: no load is issued and the value is forced to 0 (also for a pattern matrix,
        // whose value is otherwise 1).
        const int s0 = tk.pre_c + e0, s1 = tk.pre_c + e1;
        const int cbase = s0 & ~3;
        const int nchunks = s1 > s0 ? ((s1 + 3) >> 2) - (s0 >> 2) : 0;
        // edge chunk (first / last of the row): per-slot predicated gathers, masked values
        auto edge_chunk = [&](int q) {
          const int sa = cbase + 4 * q;
          const uint4 cn = lds128(col_sa + static_cast<uint32_t>(sa) * 4u);
          const uint32_t c4[4] = {cn.x, cn.y, cn.z, cn.w};
          typename RV::Raw x[4][CH];
          bool ok[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            ok[u] = sa + u >= s0 && sa + u < s1;
            const char* brow = Bl + static_cast<unsigned long long>(c4[u]) * row_bytes;
#pragma unroll
            for (int ch = 0; ch < CH; ++ch) {
              x[u][ch] = typename RV::Raw{};
              if (ok[u]) x[u][ch] = load_b<DT, VEC>(brow + (kFull ? ch * kChunkBytes : choff[ch]), pol_b);
            }
          }
          float v4[4];
          lds_vals4<ValT>(val_s0 + static_cast<uint32_t>(sa) * static_cast<uint32_t>(sizeof(ValT)), v4);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const float v = ok[u] ? v4[u] : 0.f;
#pragma unroll
            for (int ch = 0; ch < CH; ++ch) RV::fma(acc[ch], v, x[u][ch]);
          }
        };
        if (nchunks > 0) {
          if (chunk_first == 0) edge_chunk(0);
          // interior chunks 1 .. nchunks-2 are full: unpredicated, next indices prefetched.
          // Only the index-chunk address `ca` is carried through the loop (the value address is
          // derived from it) to keep the register budget for the four gathers in flight.
          const int q0 = chunk_first == 0 ? kChunkStride : chunk_first;
          uint32_t ca = col_sa + static_cast<uint32_t>(cbase + 4 * q0) * 4u;
          const uint32_t cend = col_sa + static_cast<uint32_t>(cbase + 4 * (nchunks - 1)) * 4u;
          if (ca < cend) {
            uint4 cn = lds128(ca);
            do {
              const uint32_t c4[4] = {cn.x, cn.y, cn.z, cn.w};
              typename RV::Raw x[4][CH];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const char* brow = Bl + static_cast<unsigned long long>(c4[u]) * row_bytes;
#pragma unroll
                for (int ch = 0; ch < CH; ++ch)
                  x[u][ch] = load_b<DT, VEC>(brow + (kFull ? ch * kChunkBytes : choff[ch]), pol_b);
              }
              // value chunk that pairs with index chunk `ca`
              const uint32_t va = sizeof(ValT) == 4 ? ca + (val_s0 - col_sa) : val_s0 + ((ca - col_sa) >> 1);
              ca += 16u * kChunkStride;
              if (ca < cend) cn = lds128(ca);  // next chunk's indices, while the gathers fly
              float v4[4];
              lds_vals4<ValT>(va, v4);
#pragma unroll
              for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int ch = 0; ch < CH; ++ch) RV::fma(acc[ch], v4[u], x[u][ch]);
            } while (ca < cend);
          }
          if (nchunks > 1 && ca == cend) edge_chunk(nchunks - 1);  // this group owns the last chunk
        }
      } else {
        for (int el = e0 + chunk_first; el < e1; el += kChunkStride) {
          const IdxT c = tk.scol[el];
          if (static_cast<unsigned long long>(c) >= static_cast<unsigned long long>(p.cols)) continue;
          const float v = val_at(tk.sval, el);
          const char* brow = Bl + row_offset(c, row_bytes);
#pragma unroll
          for (int ch = 0; ch < CH; ++ch)
            RV::fma(acc[ch], v, load_b<DT, VEC>(brow + (kFull ? ch * kChunkBytes : choff[ch]), pol_b));
        }
      }

      if constexpr (G > 1 && !kRowPar) {  // combine the G groups' partial rows (fixed xor tree)
#pragma unroll
        for (int off = LPR; off < 32; off <<= 1)
#pragma unroll
          for (int ch = 0; ch < CH; ++ch)
#pragma unroll
            for (int i = 0; i < VEC; ++i) acc[ch][i] += __shfl_xor_sync(0xffffffffu, acc[ch][i], off);
      }

      if (kRowPar || grp == 0) {
        if (r == re || (!kF32Out && r == rs && started_earlier)) {
          // fp32 scratch: carry[k] for the trailing partial row, head[k] for a bf16 row that
          // started in an earlier task
          float* dst = (r == re ? p.carry : p.head) + static_cast<size_t>(k) * n + col0;
#pragma unroll
          for (int ch = 0; ch < CH; ++ch)
            if (chmask & (1u << ch)) store_f32<VEC>(dst + ch * LPR * VEC, acc[ch]);
        } else {
          DT* dst = static_cast<DT*>(p.C) + static_cast<size_t>(r) * p.ldc + col0;
          if constexpr (!kF32Out) {
            if (p.flags & (kFwdAcc32In | kFwdAcc32Out)) {
              float* a32 = p.acc32 + static_cast<size_t>(r) * n + col0;
              if (p.flags & kFwdAcc32In) {
#pragma unroll
                for (int ch = 0; ch < CH; ++ch)
                  if (chmask & (1u << ch)) {
                    float o[VEC];
                    load_f32<VEC>(a32 + ch * LPR * VEC, o);
#pragma unroll
                    for (int i = 0; i < VEC; ++i) acc[ch][i] += o[i];
                  }
              }
              if (p.flags & kFwdAcc32Out) {
#pragma unroll
                for (int ch = 0; ch < CH; ++ch)
                  if (chmask & (1u << ch)) store_f32<VEC>(a32 + ch * LPR * VEC, acc[ch]);
                continue;   // next row: nothing goes to C in this pass
              }
            }
          }
          if (p.flags != 0) {
            // complete row: whole epilogue here.  Final segment of a stitched row (fp32 output
            // only — bf16 went to head[] above): fold the old C in now, the fix-up kernel adds
            // the carries and applies bias / relu.
            const bool partial = r == rs && started_earlier;
            const unsigned fl = partial ? 0u : p.flags;
#pragma unroll
            for (int ch = 0; ch < CH; ++ch)
              if (chmask & (1u << ch))
                row_epilogue<DT, VEC>(acc[ch], dst + ch * LPR * VEC, p.bias, col0 + ch * LPR * VEC, fl,
                                      (p.flags & kFwdAccumulate) != 0, static_cast<float>(e1 - e0));
          }
#pragma unroll
          for (int ch = 0; ch < CH; ++ch)
            if (chmask & (1u << ch)) RV::store_stream(dst + ch * LPR * VEC, acc[ch]);
        }
      }
    }
    t = t1;
    t1 = dynamic ? (more ? static_cast<int>(__shfl_sync(0xffffffffu, pending, 0)) : total) : t1 + total_warps;
  }
}

// Adds the carries of every row that spans several tasks, in ascending task order, on top of the
// row's final segment (a deterministic segmented reduction).  Each LANE inspects one task k: if k
// ends a row that started in an earlier task, the lane finds the first task j of that row; the
// warp then stitches the flagged rows one after another, all 32 lanes across the dense width.
template <typename DT, typename IdxT, int VEC, int WARPS, typename PartT>
__global__ void __launch_bounds__(WARPS * 32) spmm_fixup_kernel(const FwdParams p) {
  using NzT = typename PartOf<PartT>::Nz;
  using Part = PartOf<PartT>;
  const PartT* part = static_cast<const PartT*>(p.part);
  constexpr bool kF32Out = sizeof(DT) == 4;
  const int lane = threadIdx.x & 31;
  const int k = (blockIdx.x * WARPS + (threadIdx.x >> 5)) * 32 + lane;
  bool need = false;
  int j = 0, rs = 0;
  if (k >= 1 && k < p.P) {
    const PartT ps = Part::load(&part[k]);
    const int re = static_cast<int>(Part::load(&part[k + 1]).x);
    if (re > ps.x) {  // a row ends in task k
      const NzT cr = static_cast<NzT>(static_cast<const IdxT*>(p.crow)[ps.x]);
      if (cr < ps.y) {  // ... and it started before task k
        need = true;
        rs = static_cast<int>(ps.x);
        // first task holding a non-zero of the row = smallest j with part[j+1].y > cr
        j = k - 1;
        int steps = 0;
        while (j > 0 && steps < 4 && Part::load(&part[j]).y > cr) { --j; ++steps; }
        if (j > 0 && Part::load(&part[j]).y > cr) {  // hub row: finish with a binary search
          int lo = 0, hi = j;                    // invariant: part[hi].y > cr, answer in [lo, hi)
          while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (Part::load(&part[mid + 1]).y > cr) hi = mid; else lo = mid + 1;
          }
          j = lo;
        }
      }
    }
  }
  unsigned todo = __ballot_sync(0xffffffffu, need);
  const int n = p.n;
  while (todo != 0) {
    const int src = __ffs(todo) - 1;
    todo &= todo - 1;
    const int kk = __shfl_sync(0xffffffffu, k, src);
    const int jj = __shfl_sync(0xffffffffu, j, src);
    const int row = __shfl_sync(0xffffffffu, rs, src);
    DT* crow_out = static_cast<DT*>(p.C) + static_cast<size_t>(row) * p.ldc;
    for (int c0 = lane * VEC; c0 < n; c0 += 32 * VEC) {
      float sum[VEC];
#pragma unroll
      for (int i = 0; i < VEC; ++i) sum[i] = 0.f;
      for (int t = jj; t < kk; ++t) {
        float x[VEC];
        load_f32<VEC>(p.carry + static_cast<size_t>(t) * n + c0, x);
#pragma unroll
        for (int i = 0; i < VEC; ++i) sum[i] += x[i];
      }
      float h[VEC];
      if constexpr (kF32Out) {
        load_f32<VEC>(reinterpret_cast<const float*>(crow_out) + c0, h);  // already holds old C when accumulating
      } else {
        load_f32<VEC>(p.head + static_cast<size_t>(kk) * n + c0, h);
      }
#pragma unroll
      for (int i = 0; i < VEC; ++i) sum[i] += h[i];
      if constexpr (!kF32Out) {
        if (p.flags & (kFwdAcc32In | kFwdAcc32Out)) {
          float* a32 = p.acc32 + static_cast<size_t>(row) * n + c0;
          if (p.flags & kFwdAcc32In) {
            float o[VEC];
            load_f32<VEC>(a32, o);
#pragma unroll
            for (int i = 0; i < VEC; ++i) sum[i] += o[i];
          }
          if (p.flags & kFwdAcc32Out) {
            store_f32<VEC>(a32, sum);
            continue;
          }
        }
      }
      if (p.flags != 0) {
        const IdxT* crow_in = static_cast<const IdxT*>(p.crow);
        const float len = (p.flags & kFwdMean) ? static_cast<float>(static_cast<long long>(crow_in[row + 1]) -
                                                                    static_cast<long long>(crow_in[row])) : 0.f;
        row_epilogue<DT, VEC>(sum, crow_out + c0, p.bias, c0, p.flags, !kF32Out && (p.flags & kFwdAccumulate) != 0, len);
      }
      RowVec<DT, VEC>::store_stream(crow_out + c0, sum);
    }
  }
}

// part[k] = merge-path split of diagonal min(k*items, rows+nnz), k = 0..P.
template <typename IdxT, typename PartT>
__global__ void task_partition_kernel(const IdxT* __restrict__ crow, int rows, typename PartOf<PartT>::Nz nnz,
                                      int items, int P, PartT* __restrict__ part) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k > P) return;
  const long long total = static_cast<long long>(rows) + nnz;
  long long d = static_cast<long long>(k) * items;
  if (d > total) d = total;
  const long long r = merge_path_search<IdxT>(crow, rows, nnz, d);
  if constexpr (sizeof(PartT) == 8) part[k] = make_int2(static_cast<int>(r), static_cast<int>(d - r));
  else part[k] = make_longlong2(r, d - r);
}

}  // namespace ofspmm
