// Stimulus-resampling statistics of the RSA tail (rsa.cu): the Mantel permutation null of Spearman's rho and the
// stimulus bootstrap of Nili et al. 2014, for RDMs of N stimuli (P = N(N-1)/2 upper-triangle pairs).
//
// Both sort each RDM once (hba_rank_order_f64) and never again:
//   * permutation: relabelling the stimuli permutes the model's RDM entries, so its average ranks keep their
//     multiset and their moments; only the cross sum sum_{i<j} a[i,j] b[pi(i),pi(j)] changes.  Ranks enter as
//     centred doubled ranks a = 2r - (P+1), integers held in a symmetric N x N int32 matrix (diagonal 0).
//   * bootstrap: a resample with counts c_i gives every pair {i,j}, i != j, the weight w = c_i c_j (pairs of a
//     stimulus with itself are dropped).  In the RDM's fixed sorted order a tie group g of total weight W_g,
//     preceded by groups of total weight S_g, has the average rank S_g + (W_g + 1)/2 in the expanded multiset of
//     M = sum w entries - rankdata(..., 'average') of that multiset.  Centred and doubled: 2 S_g + W_g - M, which is
//     S_g + E_g - M with E_g = S_g + W_g, both read off the inclusive weight prefix in sorted order.
// Every sum is an exact int64 sum (integer atomics included), so the outputs do not depend on the order of the
// additions: bit-identical run to run.  Exact while 2 P^3 / 3 < 2^63 (N <= 2,191); the front ends check it.
#include <math_constants.h>

#include "common.cuh"
#include "rsa_keys.cuh"

namespace hba {

__host__ __device__ __forceinline__ int64_t row_start(int64_t i, int64_t N) { return i * N - i * (i + 1) / 2; }
// index of pair (i, j), i < j, in the row-major upper triangle (k = 1)
__device__ __forceinline__ int64_t pair_index(int i, int j, int N) { return row_start(i, N) + (j - i - 1); }
__device__ __forceinline__ void pair_of_index(int64_t q, int N, int& i, int& j) {
  const double b = 2.0 * N - 1.0;
  int r = (int)((b - sqrt(b * b - 8.0 * (double)q)) * 0.5);
  r = max(0, min(r, N - 2));
  while (r > 0 && row_start(r, N) > q) --r;
  while (r + 1 <= N - 2 && row_start(r + 1, N) <= q) ++r;
  i = r;
  j = (int)(q - row_start(r, N)) + r + 1;
}

static bool sums_are_exact(int64_t N) {
  const unsigned __int128 P = (unsigned __int128)(N * (N - 1) / 2);
  return 2 * P * P * P / 3 < ((unsigned __int128)1 << 63);
}

static inline int64_t align256(int64_t v) { return (v + 255) & ~(int64_t)255; }

// numpy.corrcoef's c / sqrt(d_a) / sqrt(d_b) clipped to [-1, 1]; NaN for a constant side
__device__ __forceinline__ double rho_of_sums(double sab, long long saa, long long sbb) {
  if (saa <= 0 || sbb <= 0) return CUDART_NAN;
  double r = sab / sqrt((double)saa);
  r /= sqrt((double)sbb);
  return fmin(fmax(r, -1.0), 1.0);
}

// 256-thread exclusive scan; scratch holds 9 uints; *total gets the block total (valid in every thread)
__device__ __forceinline__ unsigned int excl_scan_256(unsigned int v, unsigned int* scratch, unsigned int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  __syncthreads();
  if (lane == 31) scratch[warp] = inc;
  __syncthreads();
  unsigned int base = 0, all = 0;
#pragma unroll
  for (int w = 0; w < 8; ++w) {
    const unsigned int s = scratch[w];
    base += (w < warp) ? s : 0u;
    all += s;
  }
  *total = all;
  return base + inc - v;
}

// ------------------------------------------------------------------------------------------
// Permutation null.
//   prep: ranks [P] f64 of both RDMs -> symmetric int32 matrices A (reference), B (model) of 2r - (P+1);
//         sums[0] = sum_{i<j} a^2, sums[1] = sum_{i<j} b^2, sums[2] = number of NaN ranks
//   perm: CTA = kPermRows reference rows x kPermK permutations.  pi_p lives in shared memory for the whole CTA;
//         per row i, row pi_p(i) of B is staged in shared memory for every p, and row i of A is read once for all
//         kPermK permutations:  tot[p] += sum_j A[i,j] B[pi_p(i), pi_p(j)]  (both triangles: twice the i<j sum)
//   final: rho_p = (tot[p] / 2) / sqrt(sums[0]) / sqrt(sums[1])
constexpr int kPermK = 8;
constexpr int kPermRows = 32;
constexpr int kPermThreads = 256;

__global__ void __launch_bounds__(256)
    perm_prep_kernel(const double* __restrict__ ref_ranks, const double* __restrict__ model_ranks, int N,
                     int* __restrict__ A, int* __restrict__ B, unsigned long long* __restrict__ sums) {
  const int i = blockIdx.x;
  const double shift = (double)((int64_t)N * (N - 1) / 2 + 1);
  long long saa = 0, sbb = 0;
  unsigned int nans = 0;
  for (int j = threadIdx.x; j < N; j += 256) {
    int a = 0, b = 0;
    if (j != i) {
      const int64_t q = pair_index(min(i, j), max(i, j), N);
      const double ra = ref_ranks[q], rb = model_ranks[q];
      if (ra != ra || rb != rb) {
        ++nans;
      } else {
        a = (int)(2.0 * ra - shift);
        b = (int)(2.0 * rb - shift);
      }
    }
    A[(size_t)i * N + j] = a;
    B[(size_t)i * N + j] = b;
    if (j > i) saa += (long long)a * a, sbb += (long long)b * b;
  }
  saa = warp_sum(saa);
  sbb = warp_sum(sbb);
  nans = warp_sum(nans);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&sums[0], (unsigned long long)saa);
    atomicAdd(&sums[1], (unsigned long long)sbb);
    if (nans) atomicAdd(&sums[2], (unsigned long long)nans);
  }
}

// perms [n_perm, N] int32; a permutation with an entry outside [0, N) yields NaN (entries are clamped for the reads)
__global__ void __launch_bounds__(kPermThreads)
    perm_kernel(const int* __restrict__ A, const int* __restrict__ B, int N, const int* __restrict__ perms,
                int n_perm, unsigned long long* __restrict__ tot) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int* sB = reinterpret_cast<int*>(smem_raw);                                  // [kPermK][N]
  unsigned short* sPi = reinterpret_cast<unsigned short*>(sB + kPermK * N);  // [kPermK][N]
  __shared__ int s_bad[kPermK];
  const int p0 = blockIdx.y * kPermK;
  const int np = min(kPermK, n_perm - p0);
  if (threadIdx.x < kPermK) s_bad[threadIdx.x] = 0;
  __syncthreads();
  for (int p = 0; p < kPermK; ++p)
    for (int j = threadIdx.x; j < N; j += kPermThreads) {
      int v = p < np ? perms[(size_t)(p0 + p) * N + j] : j;
      if ((unsigned int)v >= (unsigned int)N) {
        s_bad[p] = 1;
        v = 0;
      }
      sPi[p * N + j] = (unsigned short)v;
    }
  long long acc[kPermK];
#pragma unroll
  for (int p = 0; p < kPermK; ++p) acc[p] = 0;
  const int i_end = min(N, (int)(blockIdx.x + 1) * kPermRows);
  for (int i = blockIdx.x * kPermRows; i < i_end; ++i) {
    __syncthreads();
#pragma unroll
    for (int p = 0; p < kPermK; ++p) {
      const int* row = B + (size_t)sPi[p * N + i] * N;
      for (int j = threadIdx.x; j < N; j += kPermThreads) sB[p * N + j] = row[j];
    }
    __syncthreads();
    const int* arow = A + (size_t)i * N;
    for (int j = threadIdx.x; j < N; j += kPermThreads) {
      const int a = arow[j];
#pragma unroll
      for (int p = 0; p < kPermK; ++p) acc[p] += (long long)a * sB[p * N + sPi[p * N + j]];
    }
  }
#pragma unroll
  for (int p = 0; p < kPermK; ++p) {
    const long long v = warp_sum(acc[p]);
    if ((threadIdx.x & 31) == 0 && p < np) atomicAdd(&tot[2 * (p0 + p)], (unsigned long long)v);
  }
  if (blockIdx.x == 0 && threadIdx.x < np && s_bad[threadIdx.x]) atomicAdd(&tot[2 * (p0 + threadIdx.x) + 1], 1ull);
}

__global__ void __launch_bounds__(256)
    perm_final_kernel(const unsigned long long* __restrict__ sums, const unsigned long long* __restrict__ tot,
                      int n_perm, double* __restrict__ rho) {
  const int p = blockIdx.x * 256 + threadIdx.x;
  if (p >= n_perm) return;
  if (sums[2] != 0 || tot[2 * p + 1] != 0) {
    rho[p] = CUDART_NAN;
    return;
  }
  rho[p] = rho_of_sums(0.5 * (double)(long long)tot[2 * p], (long long)sums[0], (long long)sums[1]);
}

struct PermWorkspace {
  int *A, *B;
  unsigned long long *sums, *tot;
  int64_t zero_bytes, total_bytes;
};

static PermWorkspace perm_workspace_layout(void* base, int64_t N, int64_t n_perm) {
  PermWorkspace w;
  char* p = static_cast<char*>(base);
  int64_t o = 0;
  w.A = reinterpret_cast<int*>(p + o), o += align256(N * N * 4);
  w.B = reinterpret_cast<int*>(p + o), o += align256(N * N * 4);
  const int64_t z0 = o;
  w.sums = reinterpret_cast<unsigned long long*>(p + o), o += 256;
  w.tot = reinterpret_cast<unsigned long long*>(p + o), o += align256(n_perm * 16);
  w.zero_bytes = o - z0;
  w.total_bytes = o;
  return w;
}

// ------------------------------------------------------------------------------------------
// Bootstrap.  Per RDM (reference, model a, optional model b), once per call:
//   keys:  sorted keys key[k] = f64_to_key(x[order[k]])
//   codes: pk[k] = i | NaN << 15 | j << 16 for the pair (i < j) at sorted position k; lo[k], hi[k] = first and last
//          sorted position of its tie group (binary search, as rank_final_kernel does)
// Per batch of kBootReps replicates (counts staged as uint16 in shared memory), a fixed three-phase scan over
// tiles of kBootTile sorted positions:
//   tile_sum: tsum[rep][tile] = sum of w over the tile
//   scan:     tsum[rep][.] -> exclusive tile prefix in place, M[rep] = total weight
//   prefix:   pre[rep][k] = inclusive weight prefix at sorted position k
//   rank:     v = pre[lo-1] + pre[hi] - M (= 2 S_g + W_g - M) for every pair of weight w > 0;
//             reference: scattered to pair order (aref[rep][q] = v), Saa += w v^2
//             model:     Sab += w aref[rep][q] v, Sbb += w v^2
//   final:    rho = Sab / sqrt(Saa) / sqrt(Sbb); NaN when a resampled pair of weight > 0 is NaN in any of the RDMs,
//             when a side is constant (fewer than 3 distinct stimuli included), or when the counts are not N
//             values in [0, N] summing to N
// mom[rep][8]: 0 Saa, 1 NaN / bad-count flags of the reference, 2 Sab_a, 3 Sbb_a, 4 NaN_a, 5 Sab_b, 6 Sbb_b, 7 NaN_b
constexpr int kBootReps = 8;
constexpr int kBootThreads = 256;
constexpr int kBootPer = 8;
constexpr int kBootTile = kBootThreads * kBootPer;   // 2048 sorted positions
constexpr unsigned int kPkNan = 1u << 15;

__global__ void __launch_bounds__(256)
    boot_keys_kernel(const double* __restrict__ x, const unsigned int* __restrict__ order, int64_t P,
                     unsigned long long* __restrict__ keys) {
  for (int64_t k = blockIdx.x * 256ll + threadIdx.x; k < P; k += (int64_t)gridDim.x * 256)
    keys[k] = f64_to_key(x[order[k]]);
}

__global__ void __launch_bounds__(256)
    boot_codes_kernel(const unsigned long long* __restrict__ keys, const unsigned int* __restrict__ order, int64_t P,
                      int N, unsigned int* __restrict__ pk, unsigned int* __restrict__ lo,
                      unsigned int* __restrict__ hi) {
  for (int64_t k = blockIdx.x * 256ll + threadIdx.x; k < P; k += (int64_t)gridDim.x * 256) {
    const unsigned long long key = keys[k];
    int64_t l = k, h = k;
    if (k > 0 && keys[k - 1] == key) l = lower_bound_key(keys, 0, k, key);
    if (k + 1 < P && keys[k + 1] == key) h = upper_bound_key(keys, k + 1, P, key) - 1;
    int i, j;
    pair_of_index((int64_t)order[k], N, i, j);
    pk[k] = (unsigned int)i | ((unsigned int)j << 16) | (key_is_nan(key) ? kPkNan : 0u);
    lo[k] = (unsigned int)l;
    hi[k] = (unsigned int)h;
  }
}

// flags a replicate whose counts are not N values in [0, N] summing to N
__global__ void __launch_bounds__(256)
    boot_check_counts_kernel(const int* __restrict__ counts, int N, unsigned long long* __restrict__ mom) {
  __shared__ long long scratch[32];
  const int rep = blockIdx.x;
  long long s = 0, bad = 0;
  for (int i = threadIdx.x; i < N; i += 256) {
    const int c = counts[(size_t)rep * N + i];
    s += c;
    bad += (c < 0 || c > N) ? 1 : 0;
  }
  s = block_sum(s, scratch);
  bad = block_sum(bad, scratch);
  if (threadIdx.x == 0 && (bad != 0 || s != N)) atomicAdd(&mom[(size_t)rep * 8 + 1], 1ull);
}

__device__ __forceinline__ void stage_counts(const int* __restrict__ counts, int N, int rep0, int nreps,
                                             unsigned short* sC) {
  for (int t = threadIdx.x; t < kBootReps * N; t += kBootThreads) {
    const int r = t / N;
    const int c = r < nreps ? counts[(size_t)(rep0 + r) * N + (t - r * N)] : 0;
    sC[t] = (unsigned short)min(max(c, 0), 65535);
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kBootThreads)
    boot_tile_sum_kernel(const unsigned int* __restrict__ pk, int64_t P, int N, const int* __restrict__ counts,
                         int n_boot, int tiles, unsigned int* __restrict__ tsum) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned short* sC = reinterpret_cast<unsigned short*>(smem_raw);
  __shared__ unsigned int scratch[32];
  const int rep0 = blockIdx.y * kBootReps, nreps = min(kBootReps, n_boot - rep0);
  stage_counts(counts, N, rep0, nreps, sC);
  const int64_t base = (int64_t)blockIdx.x * kBootTile + threadIdx.x * kBootPer;
  unsigned int code[kBootPer];
#pragma unroll
  for (int u = 0; u < kBootPer; ++u) code[u] = base + u < P ? pk[base + u] : 0xFFFFFFFFu;
  for (int r = 0; r < nreps; ++r) {
    const unsigned short* c = sC + r * N;
    unsigned int s = 0;
#pragma unroll
    for (int u = 0; u < kBootPer; ++u)
      if (code[u] != 0xFFFFFFFFu) s += (unsigned int)c[code[u] & 0x7FFFu] * c[code[u] >> 16];
    s = block_sum(s, scratch);
    if (threadIdx.x == 0) tsum[(size_t)(rep0 + r) * tiles + blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(kBootThreads)
    boot_tile_scan_kernel(unsigned int* __restrict__ tsum, int tiles, unsigned int* __restrict__ M) {
  __shared__ unsigned int scratch[9];
  unsigned int* t = tsum + (size_t)blockIdx.x * tiles;
  unsigned int carry = 0;
  for (int c0 = 0; c0 < tiles; c0 += kBootThreads) {
    const int idx = c0 + threadIdx.x;
    const unsigned int v = idx < tiles ? t[idx] : 0u;
    unsigned int total;
    const unsigned int ex = excl_scan_256(v, scratch, &total);
    if (idx < tiles) t[idx] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) M[blockIdx.x] = carry;
}

__global__ void __launch_bounds__(kBootThreads)
    boot_prefix_kernel(const unsigned int* __restrict__ pk, int64_t P, int N, const int* __restrict__ counts,
                       int n_boot, int tiles, const unsigned int* __restrict__ tbase, unsigned int* __restrict__ pre) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned short* sC = reinterpret_cast<unsigned short*>(smem_raw);
  __shared__ unsigned int scratch[9];
  const int rep0 = blockIdx.y * kBootReps, nreps = min(kBootReps, n_boot - rep0);
  stage_counts(counts, N, rep0, nreps, sC);
  const int64_t base = (int64_t)blockIdx.x * kBootTile + threadIdx.x * kBootPer;
  unsigned int code[kBootPer];
#pragma unroll
  for (int u = 0; u < kBootPer; ++u) code[u] = base + u < P ? pk[base + u] : 0xFFFFFFFFu;
  for (int r = 0; r < nreps; ++r) {
    const unsigned short* c = sC + r * N;
    unsigned int inc[kBootPer], s = 0;
#pragma unroll
    for (int u = 0; u < kBootPer; ++u) {
      if (code[u] != 0xFFFFFFFFu) s += (unsigned int)c[code[u] & 0x7FFFu] * c[code[u] >> 16];
      inc[u] = s;
    }
    unsigned int total;
    const unsigned int off = tbase[(size_t)(rep0 + r) * tiles + blockIdx.x] + excl_scan_256(s, scratch, &total);
    unsigned int* out = pre + (size_t)(rep0 + r) * P;
#pragma unroll
    for (int u = 0; u < kBootPer; ++u)
      if (base + u < P) out[base + u] = off + inc[u];
  }
}

template <bool kModel>
__global__ void __launch_bounds__(kBootThreads)
    boot_rank_kernel(const unsigned int* __restrict__ pk, const unsigned int* __restrict__ lo,
                     const unsigned int* __restrict__ hi, int64_t P, int N, const int* __restrict__ counts,
                     int n_boot, const unsigned int* __restrict__ pre, const unsigned int* __restrict__ M,
                     int* __restrict__ aref, unsigned long long* __restrict__ mom, int slot) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned short* sC = reinterpret_cast<unsigned short*>(smem_raw);
  const int rep0 = blockIdx.y * kBootReps, nreps = min(kBootReps, n_boot - rep0);
  stage_counts(counts, N, rep0, nreps, sC);
  unsigned int code[kBootPer], l[kBootPer], h[kBootPer];
#pragma unroll
  for (int u = 0; u < kBootPer; ++u) {
    const int64_t k = (int64_t)blockIdx.x * kBootTile + u * kBootThreads + threadIdx.x;
    const bool valid = k < P;
    code[u] = valid ? pk[k] : 0xFFFFFFFFu;
    l[u] = valid ? lo[k] : 0u;
    h[u] = valid ? hi[k] : 0u;
  }
  for (int r = 0; r < nreps; ++r) {
    const int rep = rep0 + r;
    const unsigned short* c = sC + r * N;
    const unsigned int* pr = pre + (size_t)rep * P;
    int* ar = aref + (size_t)rep * P;
    const long long m = (long long)M[rep];
    long long s0 = 0, s1 = 0, nans = 0;
#pragma unroll
    for (int u = 0; u < kBootPer; ++u) {
      if (code[u] == 0xFFFFFFFFu) continue;
      const int i = (int)(code[u] & 0x7FFFu), j = (int)(code[u] >> 16);
      const long long w = (long long)c[i] * c[j];
      if (w == 0) continue;
      const long long v = (long long)(l[u] ? pr[l[u] - 1] : 0u) + (long long)pr[h[u]] - m;
      const int64_t q = pair_index(i, j, N);
      nans += (code[u] & kPkNan) ? 1 : 0;
      if (kModel) {
        s0 += w * (long long)ar[q] * v;
        s1 += w * v * v;
      } else {
        ar[q] = (int)v;
        s0 += w * v * v;
      }
    }
    s0 = warp_sum(s0);
    s1 = warp_sum(s1);
    nans = warp_sum(nans);
    if ((threadIdx.x & 31) == 0) {
      unsigned long long* mm = mom + (size_t)rep * 8 + slot;
      if (s0) atomicAdd(&mm[0], (unsigned long long)s0);
      if (kModel && s1) atomicAdd(&mm[1], (unsigned long long)s1);
      if (nans) atomicAdd(&mm[kModel ? 2 : 1], (unsigned long long)nans);
    }
  }
}

__global__ void __launch_bounds__(256)
    boot_final_kernel(const unsigned long long* __restrict__ mom, int n_boot, double* __restrict__ rho_a,
                      double* __restrict__ rho_b) {
  const int rep = blockIdx.x * 256 + threadIdx.x;
  if (rep >= n_boot) return;
  const unsigned long long* m = mom + (size_t)rep * 8;
  const long long saa = (long long)m[0];
  rho_a[rep] = (m[1] || m[4]) ? CUDART_NAN : rho_of_sums((double)(long long)m[2], saa, (long long)m[3]);
  if (rho_b) rho_b[rep] = (m[1] || m[7]) ? CUDART_NAN : rho_of_sums((double)(long long)m[5], saa, (long long)m[6]);
}

struct BootWorkspace {
  unsigned long long* keys;
  unsigned int *pk[3], *lo[3], *hi[3];
  unsigned int *tsum, *M, *pre;
  int* aref;
  unsigned long long* mom;
  int tiles;
  int64_t total_bytes;
};

static BootWorkspace boot_workspace_layout(void* base, int64_t N, int64_t n_boot) {
  BootWorkspace w;
  const int64_t P = N * (N - 1) / 2;
  w.tiles = (int)((P + kBootTile - 1) / kBootTile);
  char* p = static_cast<char*>(base);
  int64_t o = 0;
  w.keys = reinterpret_cast<unsigned long long*>(p + o), o += align256(P * 8);
  for (int v = 0; v < 3; ++v) {
    w.pk[v] = reinterpret_cast<unsigned int*>(p + o), o += align256(P * 4);
    w.lo[v] = reinterpret_cast<unsigned int*>(p + o), o += align256(P * 4);
    w.hi[v] = reinterpret_cast<unsigned int*>(p + o), o += align256(P * 4);
  }
  w.tsum = reinterpret_cast<unsigned int*>(p + o), o += align256(n_boot * w.tiles * 4);
  w.M = reinterpret_cast<unsigned int*>(p + o), o += align256(n_boot * 4);
  w.pre = reinterpret_cast<unsigned int*>(p + o), o += align256(n_boot * P * 4);
  w.aref = reinterpret_cast<int*>(p + o), o += align256(n_boot * P * 4);
  w.mom = reinterpret_cast<unsigned long long*>(p + o), o += align256(n_boot * 64);
  w.total_bytes = o;
  return w;
}

static int boot_scan_and_rank(int v, bool model, int slot, const BootWorkspace& w, int64_t P, int N,
                              const int* counts, int n_boot, cudaStream_t s) {
  const dim3 grid(w.tiles, (n_boot + kBootReps - 1) / kBootReps);
  const size_t smem = (size_t)kBootReps * N * 2;
  boot_tile_sum_kernel<<<grid, kBootThreads, smem, s>>>(w.pk[v], P, N, counts, n_boot, w.tiles, w.tsum);
  HBA_CHECK(check_launch("boot_tile_sum_kernel"));
  boot_tile_scan_kernel<<<n_boot, kBootThreads, 0, s>>>(w.tsum, w.tiles, w.M);
  HBA_CHECK(check_launch("boot_tile_scan_kernel"));
  boot_prefix_kernel<<<grid, kBootThreads, smem, s>>>(w.pk[v], P, N, counts, n_boot, w.tiles, w.tsum, w.pre);
  HBA_CHECK(check_launch("boot_prefix_kernel"));
  if (model)
    boot_rank_kernel<true><<<grid, kBootThreads, smem, s>>>(w.pk[v], w.lo[v], w.hi[v], P, N, counts, n_boot,
                                                            w.pre, w.M, w.aref, w.mom, slot);
  else
    boot_rank_kernel<false><<<grid, kBootThreads, smem, s>>>(w.pk[v], w.lo[v], w.hi[v], P, N, counts, n_boot,
                                                             w.pre, w.M, w.aref, w.mom, slot);
  return check_launch("boot_rank_kernel");
}

}  // namespace hba

using namespace hba;

extern "C" int64_t hba_rsa_perm_workspace_bytes(int32_t N, int32_t n_perm) {
  if (N < 2 || n_perm < 1) return 0;
  return perm_workspace_layout(nullptr, N, n_perm).total_bytes;
}

extern "C" int hba_rsa_perm_null(const double* ref_ranks, const double* model_ranks, int32_t N, const int32_t* perms,
                                 int32_t n_perm, double* rho_out, void* workspace, int64_t workspace_bytes,
                                 void* stream) {
  HBA_REQUIRE(ref_ranks && model_ranks && perms && rho_out, "hba_rsa_perm_null: null pointer");
  HBA_REQUIRE(N >= 3 && sums_are_exact(N), "hba_rsa_perm_null: N=%d outside [3, 2191] (exact int64 sums)", N);
  HBA_REQUIRE(n_perm >= 1 && n_perm <= 65535 * kPermK, "hba_rsa_perm_null: n_perm=%d outside [1, %d]", n_perm,
              65535 * kPermK);
  HBA_REQUIRE(((uintptr_t)perms & 3) == 0 && ((uintptr_t)ref_ranks & 7) == 0 && ((uintptr_t)model_ranks & 7) == 0 &&
                  ((uintptr_t)rho_out & 7) == 0,
              "hba_rsa_perm_null: misaligned pointer");
  HBA_REQUIRE(workspace && workspace_bytes >= hba_rsa_perm_workspace_bytes(N, n_perm) &&
                  ((uintptr_t)workspace & 255) == 0,
              "hba_rsa_perm_null: workspace too small or not 256-byte aligned (need %lld bytes)",
              (long long)hba_rsa_perm_workspace_bytes(N, n_perm));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const PermWorkspace w = perm_workspace_layout(workspace, N, n_perm);
  const size_t smem = (size_t)kPermK * N * 6;
  static SmemAttr attr;
  HBA_CHECK(ensure_dyn_smem(perm_kernel, smem, attr, "perm_kernel"));
  cudaError_t e = cudaMemsetAsync(w.sums, 0, (size_t)w.zero_bytes, s);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("hba_rsa_perm_null: cudaMemsetAsync failed: %s", cudaGetErrorString(e));
    return HBA_ERR_CUDA;
  }
  perm_prep_kernel<<<N, 256, 0, s>>>(ref_ranks, model_ranks, N, w.A, w.B, w.sums);
  HBA_CHECK(check_launch("perm_prep_kernel"));
  perm_kernel<<<dim3((N + kPermRows - 1) / kPermRows, (n_perm + kPermK - 1) / kPermK), kPermThreads, smem, s>>>(
      w.A, w.B, N, perms, n_perm, w.tot);
  HBA_CHECK(check_launch("perm_kernel"));
  perm_final_kernel<<<(n_perm + 255) / 256, 256, 0, s>>>(w.sums, w.tot, n_perm, rho_out);
  return check_launch("perm_final_kernel");
}

extern "C" int64_t hba_rsa_boot_workspace_bytes(int32_t N, int32_t n_boot) {
  if (N < 2 || n_boot < 1) return 0;
  return boot_workspace_layout(nullptr, N, n_boot).total_bytes;
}

extern "C" int hba_rsa_bootstrap(const double* ref_tri, const uint32_t* ref_order, const double* tri_a,
                                 const uint32_t* order_a, const double* tri_b, const uint32_t* order_b, int32_t N,
                                 const int32_t* counts, int32_t n_boot, double* rho_a, double* rho_b, void* workspace,
                                 int64_t workspace_bytes, void* stream) {
  HBA_REQUIRE(ref_tri && ref_order && tri_a && order_a && counts && rho_a, "hba_rsa_bootstrap: null pointer");
  HBA_REQUIRE((tri_b == nullptr) == (order_b == nullptr) && (tri_b == nullptr) == (rho_b == nullptr),
              "hba_rsa_bootstrap: tri_b, order_b and rho_b are given together or not at all");
  HBA_REQUIRE(N >= 3 && sums_are_exact(N), "hba_rsa_bootstrap: N=%d outside [3, 2191] (exact int64 sums)", N);
  HBA_REQUIRE(n_boot >= 1 && n_boot <= 65535, "hba_rsa_bootstrap: n_boot=%d outside [1, 65535]", n_boot);
  HBA_REQUIRE(((uintptr_t)ref_tri & 7) == 0 && ((uintptr_t)tri_a & 7) == 0 && ((uintptr_t)tri_b & 7) == 0 &&
                  ((uintptr_t)ref_order & 3) == 0 && ((uintptr_t)order_a & 3) == 0 && ((uintptr_t)order_b & 3) == 0 &&
                  ((uintptr_t)counts & 3) == 0 && ((uintptr_t)rho_a & 7) == 0 && ((uintptr_t)rho_b & 7) == 0,
              "hba_rsa_bootstrap: misaligned pointer");
  HBA_REQUIRE(workspace && workspace_bytes >= hba_rsa_boot_workspace_bytes(N, n_boot) &&
                  ((uintptr_t)workspace & 255) == 0,
              "hba_rsa_bootstrap: workspace too small or not 256-byte aligned (need %lld bytes)",
              (long long)hba_rsa_boot_workspace_bytes(N, n_boot));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t P = (int64_t)N * (N - 1) / 2;
  const BootWorkspace w = boot_workspace_layout(workspace, N, n_boot);
  cudaError_t e = cudaMemsetAsync(w.mom, 0, (size_t)n_boot * 64, s);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("hba_rsa_bootstrap: cudaMemsetAsync failed: %s", cudaGetErrorString(e));
    return HBA_ERR_CUDA;
  }
  boot_check_counts_kernel<<<n_boot, 256, 0, s>>>(counts, N, w.mom);
  HBA_CHECK(check_launch("boot_check_counts_kernel"));
  const double* tri[3] = {ref_tri, tri_a, tri_b};
  const uint32_t* order[3] = {ref_order, order_a, order_b};
  const int nv = tri_b ? 3 : 2;
  int g = (int)((P + 255) / 256);
  if (g > 4 * num_sms()) g = 4 * num_sms();
  for (int v = 0; v < nv; ++v) {
    boot_keys_kernel<<<g, 256, 0, s>>>(tri[v], order[v], P, w.keys);
    HBA_CHECK(check_launch("boot_keys_kernel"));
    boot_codes_kernel<<<g, 256, 0, s>>>(w.keys, order[v], P, N, w.pk[v], w.lo[v], w.hi[v]);
    HBA_CHECK(check_launch("boot_codes_kernel"));
  }
  HBA_CHECK(boot_scan_and_rank(0, false, 0, w, P, N, counts, n_boot, s));
  for (int v = 1; v < nv; ++v) HBA_CHECK(boot_scan_and_rank(v, true, v == 1 ? 2 : 5, w, P, N, counts, n_boot, s));
  boot_final_kernel<<<(n_boot + 255) / 256, 256, 0, s>>>(w.mom, n_boot, rho_a, rho_b);
  return check_launch("boot_final_kernel");
}
