// Kendall's tau-a and tau-b of two length-n vectors (the model's and the reference's RDM triangles) from exact int64
// pair counts, by Knight's O(n log n) method:
//   1. y in its stable sorted order (y_order, from hba_rank_order_f64): the y-rank of the element at y-order position
//      p is the first position of its tie run (equal for ties, increasing across runs); the runs give n2.
//   2. x' = x[y_order] sorted stably by the radix sort of rsa.cu (rsa_radix.cuh): pairs tied in x come out in
//      ascending y.  The x runs of this order give n1, the runs equal in both x and the y-rank give n3.
//   3. D = strict inversions of the y-ranks in that order = discordant pairs, by a merge sort that counts as it
//      merges: tiles of kKtTile sorted and counted in shared memory, then one global level per doubling of the run
//      width, every CTA merging kKtTile outputs of a pair of runs split by merge path.  A right-run element counts
//      the left-run elements strictly greater than it.
//   4. S = n0 - n1 - n2 + n3 - 2 D, tau_b = S / sqrt(n0 - n1) / sqrt(n0 - n2) clipped to [-1, 1] (scipy's order of
//      operations), tau_a = S / n0.
// All counts are integer sums (integer atomics included), so outputs are bit-identical from run to run.
// n <= kKtSmallN runs all of it in one CTA (the per-epoch RSA: N = 48, n = 1,128).
#include <math_constants.h>

#include "common.cuh"
#include "rsa_keys.cuh"
#include "rsa_radix.cuh"

namespace hba {

constexpr int kKtSmallN = 2048;   // one CTA, everything in shared memory
constexpr int kKtSmallThreads = 1024;
constexpr int kKtThreads = 256;   // digit_is_constant needs 256
constexpr int kKtTile = 4096;     // elements sorted per CTA in the tile phase; outputs per CTA of a merge level
// counter block of the large path: n1, n2, n3, D, invalid-input flag
enum { kCntN1 = 0, kCntN2, kCntN3, kCntD, kCntBad, kCntWords };

template <typename K>
__device__ __forceinline__ int lower_bound_smem(const K* a, int lo, int hi, K k) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] < k) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}
template <typename K>
__device__ __forceinline__ int upper_bound_smem(const K* a, int lo, int hi, K k) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] <= k) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}
__device__ __forceinline__ int64_t lower_bound_u32(const unsigned int* __restrict__ a, int64_t lo, int64_t hi,
                                                   unsigned int k) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[mid] < k) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// Stable bottom-up merge sort of n keys (and optional payload) in shared memory, ping-ponging between buffers 0 and
// 1.  An element's place in its merged pair of runs is its index in its own run plus the number of partner-run
// elements before it: the lower bound when it comes from the left run, the upper bound from the right run, so equal
// keys keep their order.  kCount: `inv` (per thread) gets, for every right-run element, the number of left-run
// elements strictly greater than it; summed over the levels that is the number of strict inversions of the input.
// Returns the buffer holding the result.  Ends with a barrier.
template <typename K, bool kCount>
__device__ int smem_merge_sort(K* k0, K* k1, unsigned int* v0, unsigned int* v1, int n, long long& inv) {
  K* kin = k0;
  K* kout = k1;
  unsigned int* vin = v0;
  unsigned int* vout = v1;
  int which = 0;
  for (int w = 1; w < n; w <<= 1) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int start = i & ~(2 * w - 1);
      const int mid = min(start + w, n), end = min(start + 2 * w, n);
      const K key = kin[i];
      int pos;
      if (i < mid) {
        pos = i + lower_bound_smem(kin, mid, end, key) - mid;
      } else {
        const int le = upper_bound_smem(kin, start, mid, key);
        pos = (i - mid) + le;
        if (kCount) inv += mid - le;
      }
      kout[pos] = key;
      if (vin) vout[pos] = vin[i];
    }
    __syncthreads();
    K* tk = kin;
    kin = kout, kout = tk;
    unsigned int* tv = vin;
    vin = vout, vout = tv;
    which ^= 1;
  }
  return which;
}

// the outputs from the counts (one thread)
__device__ void kendall_finish(int64_t n, long long n1, long long n2, long long n3, long long D, bool invalid,
                               int64_t* counts, double* tau) {
  if (invalid) {
    counts[0] = counts[1] = counts[2] = counts[3] = -1;
    tau[0] = tau[1] = CUDART_NAN;
    return;
  }
  const long long n0 = (long long)n * (n - 1) / 2;
  const long long S = n0 - n1 - n2 + n3 - 2 * D;
  counts[0] = S, counts[1] = n1, counts[2] = n2, counts[3] = n3;
  if (n1 == n0 || n2 == n0) {
    tau[0] = tau[1] = CUDART_NAN;
    return;
  }
  double t = (double)S / sqrt((double)(n0 - n1));
  t /= sqrt((double)(n0 - n2));
  tau[0] = (double)S / (double)n0;
  tau[1] = fmin(fmax(t, -1.0), 1.0);
}

// ------------------------------------------------------------------------------------------
// n <= kKtSmallN: one CTA.  Dynamic shared memory: kx[2][n], ky[n] (later the y-ranks' merge buffers s[2][n]),
// ry[n], idx[2][n].
constexpr size_t kKtSmallSmem = (size_t)kKtSmallN * (3 * 8 + 4 + 2 * 4);

__global__ void __launch_bounds__(kKtSmallThreads)
    kendall_small_kernel(const double* __restrict__ x, const double* __restrict__ y,
                         const unsigned int* __restrict__ y_order, int n, int64_t* __restrict__ counts,
                         double* __restrict__ tau) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* kx0 = reinterpret_cast<unsigned long long*>(smem_raw);
  unsigned long long* kx1 = kx0 + kKtSmallN;
  unsigned long long* ky = kx1 + kKtSmallN;
  unsigned int* s0 = reinterpret_cast<unsigned int*>(ky);   // ky is dead once the y-ranks are known
  unsigned int* s1 = s0 + kKtSmallN;
  unsigned int* ry = reinterpret_cast<unsigned int*>(ky + kKtSmallN);
  unsigned int* i0 = ry + kKtSmallN;
  unsigned int* i1 = i0 + kKtSmallN;
  __shared__ long long scratch[32];
  int bad = 0;
  for (int p = threadIdx.x; p < n; p += kKtSmallThreads) {
    unsigned int o = y_order[p];
    if (o >= (unsigned int)n) bad = 1, o = 0;
    ky[p] = f64_to_key(y[o]);
    kx0[p] = f64_to_key(x[o]);
    i0[p] = p;
    bad |= key_is_nan(ky[p]) || key_is_nan(kx0[p]);
  }
  __syncthreads();
  long long n1 = 0, n2 = 0, n3 = 0, D = 0;
  for (int p = threadIdx.x; p < n; p += kKtSmallThreads) {
    const unsigned long long k = ky[p];
    int lo = p;
    if (p > 0) {
      bad |= ky[p - 1] > k;   // y_order does not sort y
      if (ky[p - 1] == k) lo = lower_bound_smem(ky, 0, p, k);
    }
    ry[p] = lo;
    n2 += p - lo;
  }
  bad = __syncthreads_or(bad);
  const int wx = smem_merge_sort<unsigned long long, false>(kx0, kx1, i0, i1, n, D);
  const unsigned long long* kx = wx ? kx1 : kx0;
  const unsigned int* idx = wx ? i1 : i0;
  for (int k = threadIdx.x; k < n; k += kKtSmallThreads) s0[k] = ry[idx[k]];
  __syncthreads();
  for (int k = threadIdx.x; k < n; k += kKtSmallThreads) {
    if (k > 0 && kx[k - 1] == kx[k]) {
      const int lox = lower_bound_smem(kx, 0, k, kx[k]);
      n1 += k - lox;
      if (s0[k - 1] == s0[k]) n3 += k - lower_bound_smem(s0, lox, k, s0[k]);
    }
  }
  __syncthreads();
  smem_merge_sort<unsigned int, true>(s0, s1, nullptr, nullptr, n, D);
  n1 = block_sum(n1, scratch);
  n2 = block_sum(n2, scratch);
  n3 = block_sum(n3, scratch);
  D = block_sum(D, scratch);
  if (threadIdx.x == 0) kendall_finish(n, n1, n2, n3, D, bad != 0, counts, tau);
}

// ------------------------------------------------------------------------------------------
// Large n.
// keys: ky[p] = key of y[y_order[p]], the radix sort's input keys k0[p] = key of x[y_order[p]]; flags an entry of
// y_order outside [0, n), an order that does not sort y, and NaN in x or y.
__global__ void __launch_bounds__(kKtThreads)
    kendall_keys_kernel(const double* __restrict__ x, const double* __restrict__ y,
                        const unsigned int* __restrict__ y_order, int64_t n, unsigned long long* __restrict__ ky,
                        unsigned long long* __restrict__ kx, unsigned long long* __restrict__ cnt) {
  int bad = 0;
  for (int64_t p = blockIdx.x * (int64_t)kKtThreads + threadIdx.x; p < n; p += (int64_t)gridDim.x * kKtThreads) {
    unsigned int o = y_order[p];
    if (o >= (unsigned int)n) bad = 1, o = 0;
    const unsigned long long k = f64_to_key(y[o]), kxv = f64_to_key(x[o]);
    ky[p] = k;
    kx[p] = kxv;
    bad |= key_is_nan(k) || key_is_nan(kxv);
    if (p > 0) {
      const unsigned int q = y_order[p - 1];
      bad |= q < (unsigned int)n && f64_to_key(y[q]) > k;
    }
  }
  if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(&cnt[kCntBad], 1ull);
}

// first y-order position of the tie run holding position p
__device__ __forceinline__ int64_t y_rank(const unsigned long long* __restrict__ ky, int64_t p) {
  const unsigned long long k = ky[p];
  return (p > 0 && ky[p - 1] == k) ? lower_bound_key(ky, 0, p, k) : p;
}

// after the sort: s[k] = y-rank of the element at sorted position k; n2 from the y runs
__global__ void __launch_bounds__(kKtThreads)
    kendall_ranks_kernel(const unsigned long long* __restrict__ ky, const unsigned int* __restrict__ vbuf0,
                         const unsigned int* __restrict__ vbuf1, int64_t n, const RadixCtl* __restrict__ ctl,
                         unsigned int* __restrict__ s, unsigned long long* __restrict__ cnt) {
  const int executed = radix_passes_executed(ctl, (unsigned int)n);
  const unsigned int* vals = (executed & 1) ? vbuf1 : vbuf0;
  long long n2 = 0;
  for (int64_t i = blockIdx.x * (int64_t)kKtThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kKtThreads) {
    n2 += i - y_rank(ky, i);
    s[i] = (unsigned int)y_rank(ky, executed == 0 ? i : (int64_t)vals[i]);
  }
  n2 = warp_sum(n2);
  if ((threadIdx.x & 31) == 0 && n2) atomicAdd(&cnt[kCntN2], (unsigned long long)n2);
}

// tile phase: n1 and n3 from the runs of the sorted keys and y-ranks (global reads: runs cross tiles), then the tile
// of y-ranks sorted and its inversions counted in shared memory
__global__ void __launch_bounds__(kKtThreads)
    kendall_tile_kernel(const unsigned long long* __restrict__ kbuf0, const unsigned long long* __restrict__ kbuf1,
                        int64_t n, const RadixCtl* __restrict__ ctl, const unsigned int* __restrict__ s_in,
                        unsigned int* __restrict__ s_out, unsigned long long* __restrict__ cnt) {
  __shared__ unsigned int sk[2][kKtTile];
  __shared__ long long scratch[32];
  const int executed = radix_passes_executed(ctl, (unsigned int)n);
  const unsigned long long* keys = (executed & 1) ? kbuf1 : kbuf0;
  const int64_t base = (int64_t)blockIdx.x * kKtTile;
  const int m = (int)min((int64_t)kKtTile, n - base);
  long long n1 = 0, n3 = 0, inv = 0;
  for (int j = threadIdx.x; j < m; j += kKtThreads) {
    const int64_t k = base + j;
    const unsigned int sv = s_in[k];
    sk[0][j] = sv;
    const unsigned long long kx = keys[k];
    if (k > 0 && keys[k - 1] == kx) {
      const int64_t lox = lower_bound_key(keys, 0, k, kx);
      n1 += k - lox;
      if (s_in[k - 1] == sv) n3 += k - lower_bound_u32(s_in, lox, k, sv);
    }
  }
  __syncthreads();
  const int w = smem_merge_sort<unsigned int, true>(sk[0], sk[1], nullptr, nullptr, m, inv);
  for (int j = threadIdx.x; j < m; j += kKtThreads) s_out[base + j] = sk[w][j];
  n1 = block_sum(n1, scratch);
  n3 = block_sum(n3, scratch);
  inv = block_sum(inv, scratch);
  if (threadIdx.x == 0) {
    if (n1) atomicAdd(&cnt[kCntN1], (unsigned long long)n1);
    if (n3) atomicAdd(&cnt[kCntN3], (unsigned long long)n3);
    if (inv) atomicAdd(&cnt[kCntD], (unsigned long long)inv);
  }
}

// one merge level: runs of width w (sorted) -> runs of 2w.  CTA b writes outputs [b kKtTile, (b+1) kKtTile), which lie
// in one pair of runs (2w is a multiple of kKtTile); merge path (left run first on equal keys) gives the slices of the
// two runs that produce them.  A right-run element with `le` left-run elements <= it adds (left length - le).
__global__ void __launch_bounds__(kKtThreads)
    kendall_merge_kernel(const unsigned int* __restrict__ in, unsigned int* __restrict__ out, int64_t n, int64_t w,
                         unsigned long long* __restrict__ cnt) {
  __shared__ unsigned int sm[kKtTile];
  __shared__ unsigned int so[kKtTile];
  __shared__ int64_t split[2];
  __shared__ long long scratch[32];
  const int64_t o0 = (int64_t)blockIdx.x * kKtTile;
  const int64_t ps = o0 / (2 * w) * (2 * w);
  const int64_t a_end = min(ps + w, n), b_end = min(ps + 2 * w, n);
  const int64_t la = a_end - ps, lb = b_end - a_end;
  const int64_t d0 = o0 - ps, d1 = min(d0 + kKtTile, la + lb);
  if (threadIdx.x < 2) {
    const int64_t d = threadIdx.x ? d1 : d0;
    int64_t lo = max((int64_t)0, d - lb), hi = min(d, la);
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (in[ps + mid] <= in[a_end + d - mid - 1]) lo = mid + 1;
      else hi = mid;
    }
    split[threadIdx.x] = lo;
  }
  __syncthreads();
  const int64_t a0 = split[0], b0 = d0 - a0;
  const int na = (int)(split[1] - a0), nb = (int)((d1 - split[1]) - b0);
  for (int j = threadIdx.x; j < na + nb; j += kKtThreads) sm[j] = j < na ? in[ps + a0 + j] : in[a_end + b0 + j - na];
  __syncthreads();
  long long inv = 0;
  for (int j = threadIdx.x; j < na + nb; j += kKtThreads) {
    const unsigned int v = sm[j];
    int pos;
    if (j < na) {
      pos = j + lower_bound_smem(sm, na, na + nb, v) - na;
    } else {
      const int le = upper_bound_smem(sm, 0, na, v);
      pos = (j - na) + le;
      inv += la - (a0 + le);
    }
    so[pos] = v;
  }
  __syncthreads();
  for (int j = threadIdx.x; j < na + nb; j += kKtThreads) out[ps + d0 + j] = so[j];
  inv = block_sum(inv, scratch);
  if (threadIdx.x == 0 && inv) atomicAdd(&cnt[kCntD], (unsigned long long)inv);
}

__global__ void kendall_final_kernel(const unsigned long long* __restrict__ cnt, int64_t n,
                                     int64_t* __restrict__ counts, double* __restrict__ tau) {
  kendall_finish(n, (long long)cnt[kCntN1], (long long)cnt[kCntN2], (long long)cnt[kCntN3], (long long)cnt[kCntD],
                 cnt[kCntBad] != 0, counts, tau);
}

static inline int64_t align256(int64_t v) { return (v + 255) & ~(int64_t)255; }

struct KendallWorkspace {
  RankWorkspace r;
  unsigned long long* ky;
  unsigned int *s0, *s1;
  unsigned long long* cnt;
  int64_t total_bytes;
};

static KendallWorkspace kendall_workspace_layout(void* base, int64_t n) {
  KendallWorkspace w;
  w.r = rank_workspace_layout(base, n);
  char* p = static_cast<char*>(base);
  int64_t o = align256(w.r.total_bytes);
  w.ky = reinterpret_cast<unsigned long long*>(p + o), o += align256(n * 8);
  w.s0 = reinterpret_cast<unsigned int*>(p + o), o += align256(n * 4);
  w.s1 = reinterpret_cast<unsigned int*>(p + o), o += align256(n * 4);
  w.cnt = reinterpret_cast<unsigned long long*>(p + o), o += 256;
  w.total_bytes = o;
  return w;
}

}  // namespace hba

using namespace hba;

extern "C" int64_t hba_kendall_workspace_bytes(int64_t n) {
  if (n <= kKtSmallN) return 256;
  return kendall_workspace_layout(nullptr, n).total_bytes;
}

extern "C" int hba_kendall_tau_f64(const double* x, const double* y, const uint32_t* y_order, int64_t n,
                                   int64_t* counts, double* tau, void* workspace, int64_t workspace_bytes,
                                   void* stream) {
  HBA_REQUIRE(x && y && y_order && counts && tau, "hba_kendall_tau_f64: null pointer");
  HBA_REQUIRE(n >= 2 && n < (1ll << 30), "hba_kendall_tau_f64: n=%lld outside [2, 2^30)", (long long)n);
  HBA_REQUIRE(((uintptr_t)x & 7) == 0 && ((uintptr_t)y & 7) == 0 && ((uintptr_t)y_order & 3) == 0 &&
                  ((uintptr_t)counts & 7) == 0 && ((uintptr_t)tau & 7) == 0,
              "hba_kendall_tau_f64: misaligned pointer");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (n <= kKtSmallN) {
    static SmemAttr attr;
    HBA_CHECK(ensure_dyn_smem(kendall_small_kernel, kKtSmallSmem, attr, "kendall_small_kernel"));
    kendall_small_kernel<<<1, kKtSmallThreads, kKtSmallSmem, s>>>(x, y, y_order, (int)n, counts, tau);
    return check_launch("kendall_small_kernel");
  }
  HBA_REQUIRE(workspace && workspace_bytes >= hba_kendall_workspace_bytes(n) && ((uintptr_t)workspace & 255) == 0,
              "hba_kendall_tau_f64: workspace too small or not 256-byte aligned (need %lld bytes)",
              (long long)hba_kendall_workspace_bytes(n));
  const KendallWorkspace w = kendall_workspace_layout(workspace, n);
  cudaError_t e = cudaMemsetAsync(w.cnt, 0, kCntWords * sizeof(unsigned long long), s);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("hba_kendall_tau_f64: cudaMemsetAsync failed: %s", cudaGetErrorString(e));
    return HBA_ERR_CUDA;
  }
  int g = (int)((n + kKtThreads - 1) / kKtThreads);
  if (g > 4 * num_sms()) g = 4 * num_sms();
  kendall_keys_kernel<<<g, kKtThreads, 0, s>>>(x, y, y_order, n, w.ky, w.r.k0, w.cnt);
  HBA_CHECK(check_launch("kendall_keys_kernel"));
  HBA_CHECK(radix_sort(nullptr, n, w.r, s));
  kendall_ranks_kernel<<<g, kKtThreads, 0, s>>>(w.ky, w.r.v0, w.r.v1, n, w.r.ctl, w.s0, w.cnt);
  HBA_CHECK(check_launch("kendall_ranks_kernel"));
  const int tiles = (int)((n + kKtTile - 1) / kKtTile);
  kendall_tile_kernel<<<tiles, kKtThreads, 0, s>>>(w.r.k0, w.r.k1, n, w.r.ctl, w.s0, w.s1, w.cnt);
  HBA_CHECK(check_launch("kendall_tile_kernel"));
  unsigned int *cur = w.s1, *nxt = w.s0;
  for (int64_t width = kKtTile; width < n; width *= 2) {
    kendall_merge_kernel<<<tiles, kKtThreads, 0, s>>>(cur, nxt, n, width, w.cnt);
    HBA_CHECK(check_launch("kendall_merge_kernel"));
    unsigned int* t = cur;
    cur = nxt, nxt = t;
  }
  kendall_final_kernel<<<1, 1, 0, s>>>(w.cnt, n, counts, tau);
  return check_launch("kendall_final_kernel");
}
