// bsearch.cuh — the binary search of the sampling and link-prediction kernels (sample.cu, link.cu).
#pragma once

namespace ofspmm {

// First index of the ascending a[0, n) whose value is not below x (n if there is none).
template <typename T>
__device__ __forceinline__ long long lower_bound(const T* a, long long n, T x) {
  long long lo = 0, hi = n;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (a[mid] < x) lo = mid + 1; else hi = mid;
  }
  return lo;
}

}  // namespace ofspmm
