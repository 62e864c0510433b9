// common.cuh — sm_100a device helpers shared by the ofspmm kernels: TMA bulk copy + mbarrier,
// L2 cache-policy loads/stores, 16-byte vector load/store of fp32 / bf16 rows.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

namespace ofspmm {

// ---------------------------------------------------------------- shared-memory / mbarrier / TMA

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

// Makes mbarrier.init visible to the async proxy (TMA engine) before the first bulk copy.
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}

__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}

__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}

__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}

// 1-D TMA bulk copy global -> shared (SASS: UBLKCP), completion counted in bytes on `bar`.
// dst, src 16-byte aligned; bytes a non-zero multiple of 16.
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                             uint64_t* bar, uint64_t l2_policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
      "[%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(l2_policy)
      : "memory");
}

// ---------------------------------------------------------------- element conversion

__device__ __forceinline__ float to_float(float v) { return v; }
__device__ __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }

// Value type of a pattern matrix (OFSPMM_VAL_UNIT): every stored entry is 1.0 and nothing is
// stored, staged or loaded for it.  One more ValT of the product kernels, beside float and bf16.
struct UnitVal {};
template <typename ValT> constexpr bool kIsUnit = std::is_same<ValT, UnitVal>::value;

// Value i of a value array as fp32 (1.0 for a pattern matrix, whose array pointer is null).
template <typename ValT, typename I>
__device__ __forceinline__ float val_at(const ValT* v, I i) {
  if constexpr (kIsUnit<ValT>) return 1.f;
  else return to_float(v[i]);
}

template <typename T> __device__ __forceinline__ T from_float(float v);
template <> __device__ __forceinline__ float from_float<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_float<__nv_bfloat16>(float v) {
  return __float2bfloat16_rn(v);
}

// ---------------------------------------------------------------- VEC-wide dense row access
// VEC elements of DT per lane: 16 bytes when vectorised (4 x fp32 / 8 x bf16) or 1 element.

template <typename DT, int VEC> struct RowVec;

template <> struct RowVec<float, 4> {
  using Raw = uint4;
  __device__ __forceinline__ static Raw load_raw(const float* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
  __device__ __forceinline__ static float dot(const float (&y)[4], const Raw& r, float acc) {
    acc = fmaf(y[0], __uint_as_float(r.x), acc);
    acc = fmaf(y[1], __uint_as_float(r.y), acc);
    acc = fmaf(y[2], __uint_as_float(r.z), acc);
    return fmaf(y[3], __uint_as_float(r.w), acc);
  }
  __device__ __forceinline__ static void fma(float (&acc)[4], float v, const Raw& r) {
    acc[0] = fmaf(v, __uint_as_float(r.x), acc[0]);
    acc[1] = fmaf(v, __uint_as_float(r.y), acc[1]);
    acc[2] = fmaf(v, __uint_as_float(r.z), acc[2]);
    acc[3] = fmaf(v, __uint_as_float(r.w), acc[3]);
  }
  __device__ __forceinline__ static void load(const float* p, float (&out)[4]) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p));
    out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
  }
  __device__ __forceinline__ static void store_stream(float* p, const float (&v)[4]) {
    __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
  }
};

template <> struct RowVec<float, 1> {
  using Raw = float;
  __device__ __forceinline__ static Raw load_raw(const float* p) { return __ldg(p); }
  __device__ __forceinline__ static float dot(const float (&y)[1], const Raw& r, float acc) { return fmaf(y[0], r, acc); }
  __device__ __forceinline__ static void fma(float (&acc)[1], float v, const Raw& r) { acc[0] = fmaf(v, r, acc[0]); }
  __device__ __forceinline__ static void load(const float* p, float (&out)[1]) { out[0] = __ldg(p); }
  __device__ __forceinline__ static void store_stream(float* p, const float (&v)[1]) { __stcs(p, v[0]); }
};

template <> struct RowVec<__nv_bfloat16, 8> {
  using Raw = uint4;
  __device__ __forceinline__ static Raw load_raw(const __nv_bfloat16* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
  __device__ __forceinline__ static float dot(const float (&y)[8], const Raw& r, float acc) {
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      acc = fmaf(y[2 * i], __uint_as_float(w[i] << 16), acc);
      acc = fmaf(y[2 * i + 1], __uint_as_float(w[i] & 0xffff0000u), acc);
    }
    return acc;
  }
  __device__ __forceinline__ static void fma(float (&acc)[8], float v, const Raw& r) {
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {  // bf16 -> fp32 is a 16-bit shift / mask
      acc[2 * i] = fmaf(v, __uint_as_float(w[i] << 16), acc[2 * i]);
      acc[2 * i + 1] = fmaf(v, __uint_as_float(w[i] & 0xffff0000u), acc[2 * i + 1]);
    }
  }
  __device__ __forceinline__ static void load(const __nv_bfloat16* p, float (&out)[8]) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {  // bf16 -> fp32 is a 16-bit shift
      out[2 * i] = __uint_as_float(w[i] << 16);
      out[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  __device__ __forceinline__ static void store_stream(__nv_bfloat16* p, const float (&v)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<const uint32_t*>(&h);
    }
    __stcs(reinterpret_cast<uint4*>(p), make_uint4(w[0], w[1], w[2], w[3]));
  }
};

template <> struct RowVec<__nv_bfloat16, 1> {
  using Raw = unsigned short;
  __device__ __forceinline__ static Raw load_raw(const __nv_bfloat16* p) { return __ldg(reinterpret_cast<const unsigned short*>(p)); }
  __device__ __forceinline__ static float dot(const float (&y)[1], const Raw& r, float acc) {
    return fmaf(y[0], __uint_as_float(static_cast<uint32_t>(r) << 16), acc);
  }
  __device__ __forceinline__ static void fma(float (&acc)[1], float v, const Raw& r) {
    acc[0] = fmaf(v, __uint_as_float(static_cast<uint32_t>(r) << 16), acc[0]);
  }
  __device__ __forceinline__ static void load(const __nv_bfloat16* p, float (&out)[1]) {
    out[0] = __uint_as_float(static_cast<uint32_t>(__ldg(reinterpret_cast<const unsigned short*>(p))) << 16);
  }
  __device__ __forceinline__ static void store_stream(__nv_bfloat16* p, const float (&v)[1]) {
    *p = __float2bfloat16_rn(v[0]);
  }
};

// fp32 scratch rows (carry / head partials, fp32 accumulators of multi-pass products) are stored
// as plain fp32, VEC at a time, with the streaming hint: they are written once and read once by a
// later kernel, and must not evict the dense operand from L2 on the way (cfg2: 230 MB of carries
// per launch next to a 119 MB B).
template <int VEC>
__device__ __forceinline__ void store_f32(float* p, const float (&v)[VEC]) {
  if constexpr (VEC == 4) {
    __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
  } else if constexpr (VEC == 8) {
    __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
    __stcs(reinterpret_cast<float4*>(p) + 1, make_float4(v[4], v[5], v[6], v[7]));
  } else {
#pragma unroll
    for (int i = 0; i < VEC; ++i) __stcs(p + i, v[i]);
  }
}

template <int VEC>
__device__ __forceinline__ void load_f32(const float* p, float (&v)[VEC]) {
  if constexpr (VEC == 4) {
    const float4 a = __ldcs(reinterpret_cast<const float4*>(p));
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
  } else if constexpr (VEC == 8) {
    const float4 a = __ldcs(reinterpret_cast<const float4*>(p));
    const float4 b = __ldcs(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else {
#pragma unroll
    for (int i = 0; i < VEC; ++i) v[i] = __ldcs(p + i);
  }
}

// ---------------------------------------------------------------- merge-path search
// Diagonal d of the (row-end, non-zero) merge list -> number of row-ends before it.
// Bit-exact twin of oracle/ofspmm_oracle.c:merge_path_search and of the host version in api.cu.
template <typename IdxT>
__host__ __device__ __forceinline__ int64_t merge_path_search(const IdxT* crow, int64_t rows,
                                                              int64_t nnz, int64_t d) {
  int64_t lo = d > nnz ? d - nnz : 0;
  int64_t hi = d < rows ? d : rows;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (static_cast<int64_t>(crow[mid + 1]) <= d - mid - 1) lo = mid + 1; else hi = mid;
  }
  return lo;
}

}  // namespace ofspmm
