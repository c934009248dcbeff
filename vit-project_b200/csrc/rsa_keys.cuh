// Sortable 64-bit keys of float64 values and binary searches over sorted keys, shared by the RSA tail (rsa.cu)
// and the resampling statistics (rsa_stats.cu): both must agree on the order and on what counts as a tie.
#pragma once
#include <stdint.h>

namespace hba {

// double -> uint64 whose unsigned order equals the numeric order (-0.0 canonicalised to +0.0);
// every NaN sorts above +inf
// (integer arithmetic on the two 32-bit halves: nvcc turns `bits | sign` on a reinterpreted double into the
// floating-point negation DADD -|x|, which returns the canonical NaN without the flipped sign bit)
__device__ __forceinline__ unsigned long long f64_to_key(double x) {
  x = x + 0.0;
  const int hi = __double2hiint(x), lo = __double2loint(x);
  const int neg = hi >> 31;   // all ones for a negative value
  const unsigned int khi = (unsigned int)(hi ^ (neg | (int)0x80000000)), klo = (unsigned int)(lo ^ neg);
  return ((unsigned long long)khi << 32) | klo;
}
constexpr unsigned long long kKeyPosInf = 0xFFF0000000000000ull;  // f64_to_key(+inf); NaN keys are larger
// (a negative-signed NaN maps below -inf: keys < f64_to_key(-inf) = 0x000FFFFFFFFFFFFF)
constexpr unsigned long long kKeyNegInf = 0x000FFFFFFFFFFFFFull;
__device__ __forceinline__ bool key_is_nan(unsigned long long k) { return k > kKeyPosInf || k < kKeyNegInf; }

// binary searches in the sorted key array: first index with key >= k / first index with key > k
__device__ __forceinline__ int64_t lower_bound_key(const unsigned long long* __restrict__ a, int64_t lo,
                                                   int64_t hi, unsigned long long k) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[mid] < k) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}
__device__ __forceinline__ int64_t upper_bound_key(const unsigned long long* __restrict__ a, int64_t lo,
                                                   int64_t hi, unsigned long long k) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[mid] <= k) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

}  // namespace hba
