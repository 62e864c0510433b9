/*
 * sample_key.h — the keys of neighbour sampling (include/ofspmm.h), in plain C so that the device
 * code (sample.cu) and the CPU oracle (tests/c/sample_ext_oracle.c) compute them bit for bit alike.
 *
 * Every floating-point step is one IEEE-754 correctly rounded fp64 operation (add, mul, div, fma)
 * in a fixed order, or exact bit manipulation: no libm log, no contraction.  On the device the
 * operations are the explicit round-to-nearest intrinsics; a C includer must compile with
 * -ffp-contract=off, and gets fma() from <math.h>.
 */
#ifndef OFSPMM_SAMPLE_KEY_H_
#define OFSPMM_SAMPLE_KEY_H_

#include <stdint.h>

#if defined(__CUDACC__)
#define SK_FN static __host__ __device__ __forceinline__
#else
#include <math.h>
#include <string.h>
#define SK_FN static inline
#endif

#if defined(__CUDA_ARCH__)
#define SK_ADD(a, b) __dadd_rn((a), (b))
#define SK_MUL(a, b) __dmul_rn((a), (b))
#define SK_DIV(a, b) __ddiv_rn((a), (b))
#define SK_FMA(a, b, c) __fma_rn((a), (b), (c))
#else
#define SK_ADD(a, b) ((a) + (b))
#define SK_MUL(a, b) ((a) * (b))
#define SK_DIV(a, b) ((a) / (b))
#define SK_FMA(a, b, c) fma((a), (b), (c))
#endif

SK_FN uint64_t sk_bits(double x) {
#if defined(__CUDA_ARCH__)
  return (uint64_t)__double_as_longlong(x);
#else
  uint64_t b;
  memcpy(&b, &x, sizeof b);
  return b;
#endif
}

SK_FN double sk_double(uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double((long long)b);
#else
  double x;
  memcpy(&x, &b, sizeof x);
  return x;
#endif
}

/* The sampler's 64-bit mixer: multiply by 0x9E3779B97F4A7C15, then the splitmix64 finaliser. */
SK_FN uint64_t sk_mix64(uint64_t x) {
  x *= 0x9E3779B97F4A7C15ull;
  x ^= x >> 30;
  x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27;
  x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return x;
}

/* U = ((x >> 11) + 1) * 2^-53, in (0, 1]; exact (an integer below 2^53 + 1 times a power of two). */
SK_FN double sk_uniform(uint64_t x) { return (double)((x >> 11) + 1) * 0x1p-53; }

/* -ln(u) for a normal u in (0, 1].  u = 2^k * m with m in [sqrt(2)/2, sqrt(2)); f = m - 1 is exact
 * (Sterbenz), s = f / (2 + f), and ln m = f - (f^2/2 - s (f^2/2 + R(s^2))) with the minimax R of
 * the atanh series (the classic fdlibm coefficients, error below 2^-58.45); k ln 2 is split into an
 * exactly multiplied high part and a low part.  sk_neglog(1) = +0; the tests bound the error by
 * 4 ulp against numpy.log over 10^7 inputs of the form (m + 1) 2^-53. */
SK_FN double sk_neglog(double u) {
  const double ln2_hi = 6.93147180369123816490e-01; /* 0x3FE62E42FEE00000: k * ln2_hi exact for |k| < 2^11 */
  const double ln2_lo = 1.90821492927058770002e-10; /* 0x3DEA39EF35793C76 */
  const double Lg1 = 6.666666666666735130e-01, Lg2 = 3.999999999940941908e-01, Lg3 = 2.857142874366239149e-01,
               Lg4 = 2.222219843214978396e-01, Lg5 = 1.818357216161805012e-01, Lg6 = 1.531383769920937332e-01,
               Lg7 = 1.479819860511658591e-01;
  const uint64_t b = sk_bits(u);
  const uint64_t frac = b & 0x000FFFFFFFFFFFFFull;
  int64_t k = (int64_t)(b >> 52) - 1023;
  /* mantissa bits of sqrt(2) - 1: m takes the exponent of [1/2, 1) above it, of [1, 2) below */
  const int high = frac >= 0x6A09E667F3BCDull;
  k += high;
  const double m = sk_double(frac | ((uint64_t)(high ? 1022 : 1023) << 52));
  const double f = SK_ADD(m, -1.0);
  const double s = SK_DIV(f, SK_ADD(2.0, f));
  const double z = SK_MUL(s, s);
  const double w = SK_MUL(z, z);
  const double t1 = SK_MUL(w, SK_FMA(w, SK_FMA(w, Lg6, Lg4), Lg2));
  const double t2 = SK_MUL(z, SK_FMA(w, SK_FMA(w, SK_FMA(w, Lg7, Lg5), Lg3), Lg1));
  const double R = SK_ADD(t2, t1);
  const double hfsq = SK_MUL(SK_MUL(0.5, f), f);
  const double dk = (double)k;
  /* ln u = k ln2_hi - ((hfsq - (s (hfsq + R) + k ln2_lo)) - f); negated term by term (exact) */
  const double a = SK_ADD(hfsq, -SK_FMA(s, SK_ADD(hfsq, R), SK_MUL(dk, ln2_lo)));
  return SK_ADD(SK_ADD(a, -f), SK_MUL(-dk, ln2_hi));
}

/* A weight (widened exactly to fp64) is eligible iff 0 < w < +inf: not NaN, zero, negative or infinite. */
SK_FN int sk_eligible(double w) { return w > 0.0 && w <= 0x1.fffffffffffffp+1023; }

/* The weighted key of position j: neglog(U) / w for an eligible weight, as the bits of the
 * non-negative double (order-preserving); all ones for an ineligible weight. */
SK_FN uint64_t sk_weighted_key(uint64_t x, double w) {
  if (!sk_eligible(w)) return ~0ull;
  return sk_bits(SK_DIV(sk_neglog(sk_uniform(x)), w));
}

#endif /* OFSPMM_SAMPLE_KEY_H_ */
