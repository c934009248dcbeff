// The stable LSD radix sort of (64-bit key, original index) pairs that rsa.cu builds its large-n ranking on, exposed
// to the other RSA statistics (kendall.cu) so that they sort with the same keys, passes and launch sequence.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace hba {

constexpr int kDigits = 8;

//   control block (zeroed by one memset per call):
//     hist[8][256]   global digit histograms, all eight from ONE pass over the keys
//     ticket[8]      dynamic tile numbering per pass (a tile only ever waits for tiles that already run)
//     nan_count, done  NaN detection; last-block ticket of the final reduction
struct RadixCtl {
  unsigned int hist[kDigits][256];
  unsigned int ticket[kDigits];
  unsigned int nan_count;
  unsigned int done;
  unsigned int pad[256 - kDigits - 2];
};
static_assert(sizeof(RadixCtl) == (kDigits * 256 + 256) * 4, "control block layout");

// true when digit d cannot change the order (one bin holds all n keys); needs exactly 256 threads per block
__device__ __forceinline__ bool digit_is_constant(const RadixCtl* ctl, int d, unsigned int n) {
  return __syncthreads_or(ctl->hist[d][threadIdx.x] == n) != 0;
}

// After radix_sort: the sorted keys and original indices are in buffer 1 (k1, v1) when an odd number of digit passes
// ran, in buffer 0 otherwise; when no pass ran (all keys equal) the order is the identity and v0 was never written.
__device__ __forceinline__ int radix_passes_executed(const RadixCtl* ctl, unsigned int n) {
  int executed = 0;
  for (int d = 0; d < kDigits; ++d) executed += digit_is_constant(ctl, d, n) ? 0 : 1;
  return executed;
}

struct RankWorkspace {
  unsigned long long *k0, *k1;
  unsigned int *v0, *v1;
  RadixCtl* ctl;
  unsigned int* status;
  double* partial;
  int tiles;
  int64_t zero_bytes;   // control block + status words: cleared at the start of every call
  int64_t total_bytes;
};

// layout of hba_rank_workspace_bytes(n) bytes at base (base may be null to query the size)
RankWorkspace rank_workspace_layout(void* base, int64_t n);
// Sorts n < 2^30 keys: from doubles x (f64_to_key) when x is given, else the keys already in w.k0.  Launches one
// memset, the histogram kernel and eight digit passes on s.
int radix_sort(const double* x, int64_t n, const RankWorkspace& w, cudaStream_t s);

}  // namespace hba
