// spmm_rows_kernel.cuh — whole-row SpMM for SMALL problems (one wave of warps, no long rows).
//
// The merge-path kernel (spmm_kernels.cuh) is built for throughput on large, skewed graphs: a
// partition, per-task TMA staging, carries and a fix-up launch.  On a problem the size of
// BASELINE configs[0] (4096 x 4096, 1 % dense, n = 64: 10 MFLOP) those fixed costs ARE the run
// time — three dependent launches, a staging round trip and a carry round trip per 64 items for
// ~10 us of actual gathers.  When the row-length histogram says every row is short (< 512
// non-zeros) and there are enough rows to fill the machine with one group of lanes per row, this
// kernel does the whole product in ONE launch with no workspace: a group of LPR lanes owns a row,
// reads its col / val slice LPR entries at a time (coalesced), broadcasts them inside the group
// with shuffles and gathers the dense rows four at a time, 16 bytes per lane.  Summation runs in
// storage order into one fp32 accumulator per column, exactly the order of the CPU oracle.
// Skipped (out-of-range) column indices issue no load.  Same epilogue bits as the merge kernel.
#pragma once
#include "spmm_kernels.cuh"

namespace ofspmm {

constexpr int kRowsKernelWarps = 4;

template <typename DT, typename ValT, int VEC, int LPR>
__global__ void __launch_bounds__(kRowsKernelWarps * 32)
spmm_rows_kernel(const FwdParams p) {
  constexpr int G = 32 / LPR;  // rows per warp
  constexpr bool kF32Out = sizeof(DT) == 4;
  using RV = RowVec<DT, VEC>;
  using Raw = typename RV::Raw;
  const int lane = threadIdx.x & 31;
  const int grp = lane / LPR;
  const int lig = lane % LPR;
  const int r = (blockIdx.x * kRowsKernelWarps + (threadIdx.x >> 5)) * G + grp;
  const int32_t* __restrict__ crow = static_cast<const int32_t*>(p.crow);
  const int32_t* __restrict__ col = static_cast<const int32_t*>(p.col);
  const ValT* __restrict__ val = static_cast<const ValT*>(p.val);
  const int n = p.n;
  const bool row_ok = r < p.rows;
  int beg = 0, len = 0;
  if (row_ok) {
    beg = __ldg(crow + r);
    len = __ldg(crow + r + 1) - beg;
  }
  // every lane of the warp runs the same number of iterations (full-mask shuffles below)
  int maxlen = len;
#pragma unroll
  for (int off = LPR; off < 32; off <<= 1) maxlen = max(maxlen, __shfl_xor_sync(0xffffffffu, maxlen, off));
  const bool active = lig * VEC < n;   // lanes past the dense width gather column 0 and store nothing
  const int c0 = active ? lig * VEC : 0;
  const char* __restrict__ Bc = static_cast<const char*>(p.B) + static_cast<size_t>(c0) * sizeof(DT);
  const uint32_t row_bytes = static_cast<uint32_t>(p.ldb) * sizeof(DT);
  const unsigned long long cols = static_cast<unsigned long long>(p.cols);
  float acc[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) acc[i] = 0.f;

  for (int base = 0; base < maxlen; base += LPR) {
    // this group's next LPR entries: one coalesced load each of col and val
    const int e = base + lig;
    int c = -1;      // -1: nothing to gather (past the row end, or an index outside [0, cols))
    float v = 0.f;
    if (e < len) {
      const int cc = __ldg(col + beg + e);
      if (static_cast<unsigned long long>(static_cast<long long>(cc)) < cols) {
        c = cc;
        v = val_at(val, beg + e);
      }
    }
    const int steps = min(LPR, maxlen - base);
    for (int j = 0; j < steps; j += 4) {
      int cj[4];
      float vj[4];
      Raw raw[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        // j + u < LPR always (LPR is a multiple of 4); entries past `steps` carry c = -1 anyway
        cj[u] = __shfl_sync(0xffffffffu, c, grp * LPR + j + u);
        // a pattern matrix's value is 1 wherever something is gathered (cj >= 0): nothing to send
        vj[u] = kIsUnit<ValT> ? 1.f : __shfl_sync(0xffffffffu, v, grp * LPR + j + u);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        raw[u] = Raw{};
        if (cj[u] >= 0) raw[u] = RV::load_raw(reinterpret_cast<const DT*>(Bc + row_offset<int32_t>(cj[u], row_bytes)));
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (cj[u] >= 0) RV::fma(acc, vj[u], raw[u]);
    }
  }

  if (!row_ok || !active) return;
  DT* dst = static_cast<DT*>(p.C) + static_cast<size_t>(r) * p.ldc + c0;
  if constexpr (!kF32Out) {
    if (p.flags & (kFwdAcc32In | kFwdAcc32Out)) {
      float* a32 = p.acc32 + static_cast<size_t>(r) * n + c0;
      if (p.flags & kFwdAcc32In) {
        float o[VEC];
        load_f32<VEC>(a32, o);
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[i] += o[i];
      }
      if (p.flags & kFwdAcc32Out) {
        store_f32<VEC>(a32, acc);
        return;
      }
    }
  }
  if (p.flags != 0) row_epilogue<DT, VEC>(acc, dst, p.bias, c0, p.flags, (p.flags & kFwdAccumulate) != 0, static_cast<float>(len));
  RV::store_stream(dst, acc);
}

}  // namespace ofspmm
