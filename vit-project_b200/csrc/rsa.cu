// RSA evaluation tail on the GPU (reference: behavioral_RSA, NEW:625-652, i.e. numpy.corrcoef in
// float64 + scipy.stats.spearmanr = rankdata('average') + Pearson on the ranks):
//   hba_rdm_f64       E [N, Dm] fp32 -> RDM = 1 - corrcoef(E) (f64, diag 0) and its row-major upper
//                     triangle (k=1) packed as a vector of N(N-1)/2 doubles
//   hba_rank_avg_f64  ranks with ties averaged, bit-exact w.r.t. scipy.stats.rankdata(x,'average')
//                     n <= 2048: single-CTA bitonic sort in shared memory
//                     larger n : LSD radix sort, 8-bit digits, ONE kernel per digit (decoupled look-back),
//                                all eight digit histograms from one pre-pass, constant digits skipped
//   hba_pearson_f64   two-pass (means, then centred sums) deterministic float64 reduction
//   hba_rdm_spearman  the whole chain for one checkpoint (RSA at scale, config 5): RDM entries go straight
//                     to sortable 64-bit keys, and the tie-averaged ranks are consumed by the Pearson sums
//                     in sorted order - no rank vector, no upper-triangle vector of doubles
// Bound: HBM / L2 bandwidth, no tensor-core work.  Algorithmic bytes per checkpoint (SURVEY 8d):
// 4*66*N + 40*P, P = N(N-1)/2.
#include <math_constants.h>

#include "common.cuh"
#include "rsa_keys.cuh"
#include "rsa_radix.cuh"

namespace hba {

// ------------------------------------------------------------------------------------------
// RDM: 32x32 pair tiles; each CTA centres its 64 rows in float64 (numpy.cov promotes to f64
// before subtracting the mean) and forms cov/(sd_i sd_j) exactly in numpy's order of operations:
// c = X X^T / (Dm - 1); c /= sd_i; c /= sd_j; clip to [-1, 1] (NaN kept, as numpy.clip does).
// 64 x 64 pair tiles, every thread owns a 4 x 4 micro-tile (rows ty + 16 u x columns tx + 16 w: 8 shared loads
// per 16 DFMA, bank-conflict free with the 33-double row pitch).  The 2 x 2 form on 32 x 32 tiles was bound by its
// shared-memory loads (ncu: 76 us at N = 1854 for 0.23 GFLOP of DFMA, L1 at 51 %).
// Small problems (N <= 256; the per-epoch RSA has N = 48) keep 32 x 32 tiles with 2 x 2 micro-tiles: one 64 x 64
// tile would leave a single CTA with all the work.
constexpr int kRdmChunk = 32;

template <int kRdmTile>
__global__ void __launch_bounds__(256)
    rdm_kernel(const float* __restrict__ E, int N, int Dm, double* __restrict__ rdm,
               double* __restrict__ tri, unsigned long long* __restrict__ keys) {
  constexpr int kRdmMicro = kRdmTile / 16;
  __shared__ double sX[2][kRdmTile][kRdmChunk + 1];
  __shared__ double sMean[2][kRdmTile];
  __shared__ double sSd[2][kRdmTile];
  const int bi = blockIdx.y, bj = blockIdx.x;
  if (bj < bi) return;  // upper tiles only; the lower half of rdm is written by symmetry
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int rr = warp; rr < 2 * kRdmTile; rr += 8) {
    const int side = rr / kRdmTile, r = rr % kRdmTile;
    const int row = (side == 0 ? bi : bj) * kRdmTile + r;
    double s = 0.0;
    if (row < N)
      for (int k = lane; k < Dm; k += 32) s += (double)E[(size_t)row * Dm + k];
    s = warp_sum(s);
    const double mean = s / Dm;
    double sq = 0.0;
    if (row < N)
      for (int k = lane; k < Dm; k += 32) {
        const double c = (double)E[(size_t)row * Dm + k] - mean;
        sq += c * c;
      }
    sq = warp_sum(sq);
    if (lane == 0) sMean[side][r] = mean, sSd[side][r] = sqrt(sq / (Dm - 1));
  }
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  double dot[kRdmMicro][kRdmMicro];
#pragma unroll
  for (int u = 0; u < kRdmMicro; ++u)
#pragma unroll
    for (int w = 0; w < kRdmMicro; ++w) dot[u][w] = 0.0;
  for (int k0 = 0; k0 < Dm; k0 += kRdmChunk) {
    __syncthreads();
    for (int t = threadIdx.x; t < 2 * kRdmTile * kRdmChunk; t += 256) {
      const int side = t / (kRdmTile * kRdmChunk), r = (t / kRdmChunk) % kRdmTile, k = t % kRdmChunk;
      const int row = (side == 0 ? bi : bj) * kRdmTile + r;
      sX[side][r][k] = (row < N && k0 + k < Dm)
                           ? (double)E[(size_t)row * Dm + k0 + k] - sMean[side][r]
                           : 0.0;
    }
    __syncthreads();
    const int kn = min(kRdmChunk, Dm - k0);
#pragma unroll 4
    for (int k = 0; k < kn; ++k) {
      double a[kRdmMicro], b[kRdmMicro];
#pragma unroll
      for (int u = 0; u < kRdmMicro; ++u) a[u] = sX[0][ty + 16 * u][k], b[u] = sX[1][tx + 16 * u][k];
#pragma unroll
      for (int u = 0; u < kRdmMicro; ++u)
#pragma unroll
        for (int w = 0; w < kRdmMicro; ++w) dot[u][w] += a[u] * b[w];
    }
  }
#pragma unroll
  for (int u = 0; u < kRdmMicro; ++u)
#pragma unroll
    for (int w = 0; w < kRdmMicro; ++w) {
      const int a = ty + 16 * u, b = tx + 16 * w;
      const int i = bi * kRdmTile + a, j = bj * kRdmTile + b;
      if (i >= N || j >= N || j < i) continue;
      double c = dot[u][w] / (Dm - 1);
      c /= sSd[0][a];
      c /= sSd[1][b];
      c = (c != c) ? c : fmin(fmax(c, -1.0), 1.0);   // CUDA fmin/fmax would drop a NaN; numpy.clip keeps it
      const double v = (i == j) ? 0.0 : 1.0 - c;
      if (rdm) {
        rdm[(size_t)i * N + j] = v;
        rdm[(size_t)j * N + i] = v;
      }
      if (j > i) {
        const size_t p = (size_t)i * N - (size_t)i * (i + 1) / 2 + (j - i - 1);
        if (tri) tri[p] = v;
        if (keys) keys[p] = f64_to_key(v);
      }
    }
}

// single CTA: bitonic sort of up to 2048 (key, index) pairs in shared memory, tie-run averaging.
// Any NaN makes every rank NaN (scipy.stats.rankdata, nan_policy='propagate').  kOrder: also writes the stable
// sorted order (order[p] = index of the p-th smallest key, NaN keys at the ends), which needs the sort even with NaN.
constexpr int kSmallN = 2048;
template <bool kOrder>
__global__ void __launch_bounds__(1024)
    rank_small_kernel(const double* __restrict__ x, int n, double* __restrict__ ranks,
                      unsigned int* __restrict__ order) {
  __shared__ unsigned long long sk[kSmallN];
  __shared__ unsigned short si[kSmallN];
  int has_nan = 0;
  for (int i = threadIdx.x; i < kSmallN; i += 1024) {
    const double v = (i < n) ? x[i] : 0.0;
    has_nan |= (v != v);
    sk[i] = (i < n) ? f64_to_key(v) : ~0ull;  // padding sorts last (index breaks the tie)
    si[i] = (unsigned short)i;
  }
  has_nan = __syncthreads_or(has_nan);
  if (!kOrder && has_nan) {
    for (int i = threadIdx.x; i < n; i += 1024) ranks[i] = CUDART_NAN;
    return;
  }
  for (int k = 2; k <= kSmallN; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < kSmallN; i += 1024) {
        const int l = i ^ j;
        if (l > i) {
          const bool up = ((i & k) == 0);
          const unsigned long long a = sk[i], b = sk[l];
          const unsigned short ia = si[i], ib = si[l];
          const bool gt = (a > b) || (a == b && ia > ib);
          if (gt == up) {
            sk[i] = b, sk[l] = a;
            si[i] = ib, si[l] = ia;
          }
        }
      }
      __syncthreads();
    }
  }
  // positions [0, n) now hold the real elements (padding has the largest key or index)
  if (kOrder) {
    for (int p = threadIdx.x; p < n; p += 1024) order[p] = si[p];
    if (has_nan) {
      for (int i = threadIdx.x; i < n; i += 1024) ranks[i] = CUDART_NAN;
      return;
    }
  }
  for (int p = threadIdx.x; p < n; p += 1024) {
    if (p == 0 || sk[p] != sk[p - 1]) {
      int e = p;
      while (e + 1 < n && sk[e + 1] == sk[p]) ++e;
      const double r = 0.5 * (double)(p + e) + 1.0;
      for (int q = p; q <= e; ++q) ranks[si[q]] = r;
    }
  }
}

// ------------------------------------------------------------------------------------------
// Large n: least-significant-digit radix sort of (key, original index) pairs (control block: rsa_radix.cuh).
//     status[8][tiles][256]  decoupled look-back words: flag (2 bits) | count (30 bits)
//   A digit whose histogram has a single non-empty bin leaves the order unchanged: its pass returns at once
//   (RDM entries live in [0, 2]: the top byte is constant).  Every CTA derives which buffer holds the current
//   order from the histograms themselves (number of passes executed before it), so no extra state is needed and
//   the launch sequence is fixed (CUDA-graph friendly).
constexpr int kRadixThreads = 256;
constexpr int kRadixWarps = kRadixThreads / 32;
// 8 elements per thread: with 16 the pass kernel needed 128 registers (2 CTAs = 16 warps per SM) and was bound by
// the latency of its shared-memory / shuffle chain (ncu: 19 % issue-active, 38 us per pass at 1.7 M keys)
constexpr int kRadixIters = 8;                                   // per warp
constexpr int kRadixTile = kRadixWarps * kRadixIters * 32;       // 2048 elements per CTA
constexpr unsigned int kFlagAgg = 1u << 30, kFlagIncl = 2u << 30, kCountMask = (1u << 30) - 1u;

// keys (from doubles, or already produced by rdm_kernel) + all eight digit histograms + NaN count
__global__ void __launch_bounds__(256)
    radix_hist_kernel(const double* __restrict__ x, unsigned long long* __restrict__ keys, int64_t n,
                      RadixCtl* __restrict__ ctl) {
  __shared__ unsigned int sh[kDigits][256];
  for (int i = threadIdx.x; i < kDigits * 256; i += 256) (&sh[0][0])[i] = 0;
  __syncthreads();
  unsigned int nans = 0;
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    unsigned long long k;
    if (x) {
      k = f64_to_key(x[i]);
      keys[i] = k;
    } else {
      k = keys[i];
    }
    nans += key_is_nan(k) ? 1u : 0u;
#pragma unroll
    for (int d = 0; d < kDigits; ++d) {
      const unsigned int digit = (unsigned int)(k >> (8 * d)) & 0xffu;
      // warp-aggregated when the whole warp agrees (the constant high digits), plain shared atomics otherwise
      int all_same;
      __match_all_sync(__activemask(), digit, &all_same);
      if (all_same) {
        const unsigned int act = __activemask();
        if ((threadIdx.x & 31) == (__ffs(act) - 1)) atomicAdd(&sh[d][digit], __popc(act));
      } else {
        atomicAdd(&sh[d][digit], 1u);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kDigits * 256; i += 256) {
    const unsigned int c = (&sh[0][0])[i];
    if (c) atomicAdd(&ctl->hist[0][0] + i, c);
  }
  nans = warp_sum(nans);
  if ((threadIdx.x & 31) == 0 && nans) atomicAdd(&ctl->nan_count, nans);
}

// block-wide exclusive scan of one value per thread (256 threads); `scratch` holds 8 uints
__device__ __forceinline__ unsigned int block_excl_scan_256(unsigned int v, unsigned int* scratch) {
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
  unsigned int base = 0;
#pragma unroll
  for (int w = 0; w < kRadixWarps; ++w)
    if (w < warp) base += scratch[w];
  return base + inc - v;
}

__global__ void __launch_bounds__(kRadixThreads, 4)
    radix_pass_kernel(unsigned long long* __restrict__ kbuf0, unsigned long long* __restrict__ kbuf1,
                      unsigned int* __restrict__ vbuf0, unsigned int* __restrict__ vbuf1, int64_t n, int pass,
                      RadixCtl* __restrict__ ctl, unsigned int* __restrict__ status_all, int num_tiles) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* s_keys = reinterpret_cast<unsigned long long*>(smem_raw);           // [kRadixTile]
  unsigned int* s_vals = reinterpret_cast<unsigned int*>(s_keys + kRadixTile);            // [kRadixTile]
  unsigned int (*warp_hist)[256] = reinterpret_cast<unsigned int (*)[256]>(s_vals + kRadixTile);  // [8][256]
  unsigned int* s_local = &warp_hist[0][0] + kRadixWarps * 256;                           // [256] first local index of a bin
  int* s_gbase = reinterpret_cast<int*>(s_local + 256);                                   // [256] global pos - local idx
  unsigned int* s_scratch = reinterpret_cast<unsigned int*>(s_gbase + 256);               // [8] + tile
  const unsigned int n32 = (unsigned int)n;
  if (digit_is_constant(ctl, pass, n32)) return;
  int executed_before = 0;
  for (int d = 0; d < pass; ++d) executed_before += digit_is_constant(ctl, d, n32) ? 0 : 1;
  const bool flip = executed_before & 1;
  const unsigned long long* keys_in = flip ? kbuf1 : kbuf0;
  unsigned long long* keys_out = flip ? kbuf0 : kbuf1;
  const unsigned int* vals_in = flip ? vbuf1 : vbuf0;
  unsigned int* vals_out = flip ? vbuf0 : vbuf1;
  const bool implicit_vals = executed_before == 0;   // the first executed pass: value = original index

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) s_scratch[kRadixWarps] = atomicAdd(&ctl->ticket[pass], 1u);
  for (int b = lane; b < 256; b += 32) warp_hist[warp][b] = 0;
  __syncthreads();
  const int tile = (int)s_scratch[kRadixWarps];
  const int shift = 8 * pass;
  const int64_t tbase = (int64_t)tile * kRadixTile;
  const int64_t wbase = tbase + (int64_t)warp * kRadixIters * 32;

  // ---- load + rank inside the warp (element order = (warp, iteration, lane): stable) ----
  unsigned long long key[kRadixIters];
  unsigned int val[kRadixIters];
  unsigned short off[kRadixIters];
#pragma unroll
  for (int it = 0; it < kRadixIters; ++it) {
    const int64_t idx = wbase + it * 32 + lane;
    const bool valid = idx < n;
    key[it] = valid ? keys_in[idx] : ~0ull;
    val[it] = valid ? (implicit_vals ? (unsigned int)idx : vals_in[idx]) : 0u;
  }
#pragma unroll
  for (int it = 0; it < kRadixIters; ++it) {
    const bool valid = wbase + it * 32 + lane < n;
    const unsigned int digit = valid ? (unsigned int)(key[it] >> shift) & 0xffu : 0x100u;
    const unsigned int peers = __match_any_sync(0xffffffffu, digit);
    const unsigned int rank = __popc(peers & ((1u << lane) - 1u));
    unsigned int base = 0;
    if (valid) base = warp_hist[warp][digit];
    __syncwarp();
    if (valid && rank == 0) warp_hist[warp][digit] = base + __popc(peers);
    __syncwarp();
    off[it] = (unsigned short)(base + rank);
  }
  __syncthreads();

  // ---- per bin (thread b = bin b): warp prefixes, tile count, look-back over the preceding tiles ----
  {
    const int b = threadIdx.x;
    unsigned int run = 0;
#pragma unroll
    for (int w = 0; w < kRadixWarps; ++w) {
      const unsigned int c = warp_hist[w][b];
      warp_hist[w][b] = run;
      run += c;
    }
    volatile unsigned int* status = status_all + ((size_t)pass * num_tiles) * 256;
    status[(size_t)tile * 256 + b] = (tile == 0 ? kFlagIncl : kFlagAgg) | run;
    const unsigned int local_start = block_excl_scan_256(run, s_scratch);
    const unsigned int global_start = block_excl_scan_256(ctl->hist[pass][b], s_scratch);
    unsigned int excl = 0;
    for (int p = tile - 1; p >= 0; --p) {
      unsigned int s;
      do {
        s = status[(size_t)p * 256 + b];
      } while ((s >> 30) == 0u);
      excl += s & kCountMask;
      if ((s >> 30) == 2u) break;
    }
    if (tile > 0) status[(size_t)tile * 256 + b] = kFlagIncl | (excl + run);
    s_local[b] = local_start;
    s_gbase[b] = (int)(global_start + excl) - (int)local_start;
  }
  __syncthreads();

  // ---- reorder inside the tile (shared memory), then write runs of equal digits contiguously ----
#pragma unroll
  for (int it = 0; it < kRadixIters; ++it) {
    if (wbase + it * 32 + lane < n) {
      const unsigned int digit = (unsigned int)(key[it] >> shift) & 0xffu;
      const unsigned int li = s_local[digit] + warp_hist[warp][digit] + off[it];
      s_keys[li] = key[it];
      s_vals[li] = val[it];
    }
  }
  __syncthreads();
  const int valid_count = (int)min((int64_t)kRadixTile, n - tbase);
#pragma unroll 4
  for (int i = threadIdx.x; i < valid_count; i += kRadixThreads) {
    const unsigned long long k = s_keys[i];
    const unsigned int digit = (unsigned int)(k >> shift) & 0xffu;
    const int64_t pos = (int64_t)s_gbase[digit] + i;
    keys_out[pos] = k;
    vals_out[pos] = s_vals[i];
  }
}
constexpr size_t kRadixPassSmem = (size_t)kRadixTile * 12 + (kRadixWarps * 256 + 256 + 256 + 16) * 4;

// After the sort.  Position p of the sorted order holds (key, original index v); its rank is the mean of the
// 1-based positions of its tie run (found by binary search, so that even an all-equal input costs O(log n) per
// element).  ranks_out (optional): ranks[v] = rank.  ref (optional): Pearson sums of (rank, ref[v]) about the
// exact mean (n+1)/2 of any average-rank vector; the last CTA adds the partials in a fixed order and writes
// rho = Sab / sqrt(Saa) / sqrt(Sbb) clipped to [-1, 1] (numpy.corrcoef), NaN when any input was NaN or constant.
constexpr int kFinalBlocks = 592;
__global__ void __launch_bounds__(256)
    rank_final_kernel(const unsigned long long* __restrict__ kbuf0, const unsigned long long* __restrict__ kbuf1,
                      const unsigned int* __restrict__ vbuf0, const unsigned int* __restrict__ vbuf1, int64_t n,
                      RadixCtl* __restrict__ ctl, double* __restrict__ ranks_out, const double* __restrict__ ref,
                      double* __restrict__ partial, double* __restrict__ rho) {
  __shared__ double scratch[32];
  __shared__ int s_last;
  const unsigned int n32 = (unsigned int)n;
  const int executed = radix_passes_executed(ctl, n32);
  const unsigned long long* keys = (executed & 1) ? kbuf1 : kbuf0;
  const unsigned int* vals = (executed & 1) ? vbuf1 : vbuf0;
  const bool implicit_vals = executed == 0;
  const bool any_nan = ctl->nan_count != 0;
  const double mu = 0.5 * (double)(n + 1);
  double sab = 0.0, saa = 0.0, sbb = 0.0;
  for (int64_t p = blockIdx.x * 256ll + threadIdx.x; p < n; p += (int64_t)gridDim.x * 256) {
    const unsigned long long k = keys[p];
    const bool tie_left = p > 0 && keys[p - 1] == k;
    const bool tie_right = p + 1 < n && keys[p + 1] == k;
    int64_t lo = p, hi = p;
    if (tie_left) lo = lower_bound_key(keys, 0, p, k);
    if (tie_right) hi = upper_bound_key(keys, p + 1, n, k) - 1;
    const double r = any_nan ? CUDART_NAN : 0.5 * (double)(lo + hi) + 1.0;
    const unsigned int v = implicit_vals ? (unsigned int)p : vals[p];
    if (ranks_out) ranks_out[v] = r;
    if (ref) {
      const double da = r - mu, db = ref[v] - mu;
      sab += da * db, saa += da * da, sbb += db * db;
    }
  }
  if (!ref) return;
  sab = block_sum(sab, scratch);
  saa = block_sum(saa, scratch);
  sbb = block_sum(sbb, scratch);
  if (threadIdx.x == 0) {
    partial[blockIdx.x] = sab;
    partial[kFinalBlocks + blockIdx.x] = saa;
    partial[2 * kFinalBlocks + blockIdx.x] = sbb;
    __threadfence();
    s_last = (atomicAdd(&ctl->done, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  double t[3] = {0.0, 0.0, 0.0};
  for (int i = threadIdx.x; i < (int)gridDim.x; i += 256) {
    t[0] += *reinterpret_cast<volatile double*>(partial + i);
    t[1] += *reinterpret_cast<volatile double*>(partial + kFinalBlocks + i);
    t[2] += *reinterpret_cast<volatile double*>(partial + 2 * kFinalBlocks + i);
  }
  t[0] = block_sum(t[0], scratch);
  t[1] = block_sum(t[1], scratch);
  t[2] = block_sum(t[2], scratch);
  if (threadIdx.x == 0) {
    double r = t[0] / sqrt(t[1]);
    r /= sqrt(t[2]);
    *rho = (r != r) ? r : fmin(fmax(r, -1.0), 1.0);
  }
}

// After the sort: the stable sorted order (original index of every sorted position) out of whichever value buffer
// the executed passes left it in; identity when no digit pass ran (all keys equal).
__global__ void __launch_bounds__(256)
    sorted_order_kernel(const unsigned int* __restrict__ vbuf0, const unsigned int* __restrict__ vbuf1, int64_t n,
                        RadixCtl* __restrict__ ctl, unsigned int* __restrict__ order) {
  const unsigned int n32 = (unsigned int)n;
  const int executed = radix_passes_executed(ctl, n32);
  const unsigned int* vals = (executed & 1) ? vbuf1 : vbuf0;
  for (int64_t p = blockIdx.x * 256ll + threadIdx.x; p < n; p += (int64_t)gridDim.x * 256)
    order[p] = executed == 0 ? (unsigned int)p : vals[p];
}

// ------------------------------------------------------------------------------------------
// Pearson correlation in float64: pass 1 partial sums -> means; pass 2 centred partial sums;
// finalize in a fixed order (deterministic).  ws: [0,1024) sum a, [1024,2048) sum b,
// [2048,3072) Sab, [3072,4096) Saa, [4096,5120) Sbb.
constexpr int kPearsonBlocks = 1024;

__global__ void __launch_bounds__(256)
    pearson_sums_kernel(const double* __restrict__ a, const double* __restrict__ b, int64_t n,
                        double* __restrict__ ws) {
  __shared__ double scratch[32];
  double sa = 0.0, sb = 0.0;
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    sa += a[i];
    sb += b[i];
  }
  sa = block_sum(sa, scratch);
  sb = block_sum(sb, scratch);
  if (threadIdx.x == 0) ws[blockIdx.x] = sa, ws[kPearsonBlocks + blockIdx.x] = sb;
}

__global__ void __launch_bounds__(256)
    pearson_centered_kernel(const double* __restrict__ a, const double* __restrict__ b, int64_t n,
                            int nblocks, double* __restrict__ ws) {
  __shared__ double scratch[32];
  __shared__ double means[2];
  if (threadIdx.x == 0) {
    double sa = 0.0, sb = 0.0;
    for (int i = 0; i < nblocks; ++i) sa += ws[i], sb += ws[kPearsonBlocks + i];
    means[0] = sa / (double)n, means[1] = sb / (double)n;
  }
  __syncthreads();
  const double ma = means[0], mb = means[1];
  double sab = 0.0, saa = 0.0, sbb = 0.0;
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    const double da = a[i] - ma, db = b[i] - mb;
    sab += da * db, saa += da * da, sbb += db * db;
  }
  sab = block_sum(sab, scratch);
  saa = block_sum(saa, scratch);
  sbb = block_sum(sbb, scratch);
  if (threadIdx.x == 0) {
    ws[2 * kPearsonBlocks + blockIdx.x] = sab;
    ws[3 * kPearsonBlocks + blockIdx.x] = saa;
    ws[4 * kPearsonBlocks + blockIdx.x] = sbb;
  }
}

__global__ void pearson_final_kernel(const double* __restrict__ ws, int nblocks,
                                     double* __restrict__ rho) {
  double sab = 0.0, saa = 0.0, sbb = 0.0;
  for (int i = 0; i < nblocks; ++i) {
    sab += ws[2 * kPearsonBlocks + i];
    saa += ws[3 * kPearsonBlocks + i];
    sbb += ws[4 * kPearsonBlocks + i];
  }
  // numpy.corrcoef: c / sqrt(d_a) / sqrt(d_b), clipped to [-1, 1]; a NaN (constant or NaN input) stays NaN
  double r = sab / sqrt(saa);
  r /= sqrt(sbb);
  *rho = (r != r) ? r : fmin(fmax(r, -1.0), 1.0);
}

static inline int64_t align256(int64_t v) { return (v + 255) & ~(int64_t)255; }

RankWorkspace rank_workspace_layout(void* base, int64_t n) {
  RankWorkspace w;
  w.tiles = (int)((n + kRadixTile - 1) / kRadixTile);
  char* p = static_cast<char*>(base);
  int64_t o = 0;
  w.k0 = reinterpret_cast<unsigned long long*>(p + o), o += align256(n * 8);
  w.k1 = reinterpret_cast<unsigned long long*>(p + o), o += align256(n * 8);
  w.v0 = reinterpret_cast<unsigned int*>(p + o), o += align256(n * 4);
  w.v1 = reinterpret_cast<unsigned int*>(p + o), o += align256(n * 4);
  w.partial = reinterpret_cast<double*>(p + o), o += align256(3 * kFinalBlocks * 8);
  const int64_t z0 = o;
  w.ctl = reinterpret_cast<RadixCtl*>(p + o), o += (int64_t)sizeof(RadixCtl);
  w.status = reinterpret_cast<unsigned int*>(p + o), o += align256((int64_t)kDigits * w.tiles * 256 * 4);
  w.zero_bytes = o - z0;
  w.total_bytes = o + 256;
  return w;
}

int radix_sort(const double* x, int64_t n, const RankWorkspace& w, cudaStream_t s) {
  static SmemAttr attr;
  HBA_CHECK(ensure_dyn_smem(radix_pass_kernel, kRadixPassSmem, attr, "radix_pass_kernel"));
  cudaError_t e = cudaMemsetAsync(w.ctl, 0, (size_t)w.zero_bytes, s);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("rank: cudaMemsetAsync failed: %s", cudaGetErrorString(e));
    return HBA_ERR_CUDA;
  }
  int g = (int)((n + 256 * 8 - 1) / (256 * 8));
  if (g > 2 * num_sms()) g = 2 * num_sms();
  radix_hist_kernel<<<g, 256, 0, s>>>(x, w.k0, n, w.ctl);
  HBA_CHECK(check_launch("radix_hist_kernel"));
  for (int pass = 0; pass < kDigits; ++pass) {
    radix_pass_kernel<<<w.tiles, kRadixThreads, kRadixPassSmem, s>>>(w.k0, w.k1, w.v0, w.v1, n, pass, w.ctl,
                                                                     w.status, w.tiles);
    HBA_CHECK(check_launch("radix_pass_kernel"));
  }
  return HBA_OK;
}

// sort + final pass; keys must already be in w.k0 unless x is given
static int rank_large(const double* x, int64_t n, const RankWorkspace& w, double* ranks_out, const double* ref,
                      double* rho, cudaStream_t s) {
  HBA_CHECK(radix_sort(x, n, w, s));
  int fb = (int)((n + 255) / 256);
  if (fb > kFinalBlocks) fb = kFinalBlocks;
  rank_final_kernel<<<fb, 256, 0, s>>>(w.k0, w.k1, w.v0, w.v1, n, w.ctl, ranks_out, ref, w.partial, rho);
  return check_launch("rank_final_kernel");
}

static void launch_rdm(const float* E, int N, int Dm, double* rdm, double* tri, unsigned long long* keys,
                       cudaStream_t s) {
  if (N <= 256) {
    const int nb = (N + 31) / 32;
    rdm_kernel<32><<<dim3(nb, nb), 256, 0, s>>>(E, N, Dm, rdm, tri, keys);
  } else {
    const int nb = (N + 63) / 64;
    rdm_kernel<64><<<dim3(nb, nb), 256, 0, s>>>(E, N, Dm, rdm, tri, keys);
  }
}

}  // namespace hba

using namespace hba;

extern "C" int hba_rdm_f64(const float* E, int32_t N, int32_t Dm, double* rdm, double* tri,
                           void* stream) {
  HBA_REQUIRE(E && (rdm || tri) && N > 1, "hba_rdm_f64: bad arguments");
  HBA_REQUIRE(Dm > 1, "hba_rdm_f64: Dm=%d must be > 1", Dm);
  launch_rdm(E, N, Dm, rdm, tri, nullptr, static_cast<cudaStream_t>(stream));
  return check_launch("rdm_kernel");
}

extern "C" int64_t hba_rank_workspace_bytes(int64_t n) {
  if (n <= kSmallN) return 256;
  return rank_workspace_layout(nullptr, n).total_bytes;
}

extern "C" int hba_rank_avg_f64(const double* x, int64_t n, double* ranks, void* workspace,
                                int64_t workspace_bytes, void* stream) {
  HBA_REQUIRE(x && ranks && n > 0, "hba_rank_avg_f64: bad arguments");
  HBA_REQUIRE(n < (1ll << 30), "hba_rank_avg_f64: n too large");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (n <= kSmallN) {
    rank_small_kernel<false><<<1, 1024, 0, s>>>(x, (int)n, ranks, nullptr);
    return check_launch("rank_small_kernel");
  }
  HBA_REQUIRE(workspace && workspace_bytes >= hba_rank_workspace_bytes(n) &&
                  ((uintptr_t)workspace & 255) == 0,
              "hba_rank_avg_f64: workspace too small or not 256-byte aligned (need %lld bytes)",
              (long long)hba_rank_workspace_bytes(n));
  return rank_large(x, n, rank_workspace_layout(workspace, n), ranks, nullptr, nullptr, s);
}

extern "C" int hba_rank_order_f64(const double* x, int64_t n, uint32_t* order, double* ranks, void* workspace,
                                  int64_t workspace_bytes, void* stream) {
  HBA_REQUIRE(x && order && ranks && n > 0, "hba_rank_order_f64: bad arguments");
  HBA_REQUIRE(n < (1ll << 30), "hba_rank_order_f64: n too large");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (n <= kSmallN) {
    rank_small_kernel<true><<<1, 1024, 0, s>>>(x, (int)n, ranks, order);
    return check_launch("rank_small_kernel");
  }
  HBA_REQUIRE(workspace && workspace_bytes >= hba_rank_workspace_bytes(n) &&
                  ((uintptr_t)workspace & 255) == 0,
              "hba_rank_order_f64: workspace too small or not 256-byte aligned (need %lld bytes)",
              (long long)hba_rank_workspace_bytes(n));
  const RankWorkspace w = rank_workspace_layout(workspace, n);
  HBA_CHECK(rank_large(x, n, w, ranks, nullptr, nullptr, s));
  int g = (int)((n + 255) / 256);
  if (g > kFinalBlocks) g = kFinalBlocks;
  sorted_order_kernel<<<g, 256, 0, s>>>(w.v0, w.v1, n, w.ctl, order);
  return check_launch("sorted_order_kernel");
}

extern "C" int hba_pearson_f64(const double* a, const double* b, int64_t n, double* rho_out,
                               double* workspace, void* stream) {
  HBA_REQUIRE(a && b && rho_out && workspace && n > 1, "hba_pearson_f64: bad arguments");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int nblocks = (int)((n + 255) / 256);
  if (nblocks > kPearsonBlocks) nblocks = kPearsonBlocks;
  pearson_sums_kernel<<<nblocks, 256, 0, s>>>(a, b, n, workspace);
  pearson_centered_kernel<<<nblocks, 256, 0, s>>>(a, b, n, nblocks, workspace);
  pearson_final_kernel<<<1, 1, 0, s>>>(workspace, nblocks, rho_out);
  return check_launch("pearson kernels");
}

extern "C" int hba_rdm_spearman(const float* E, int32_t N, int32_t Dm, const double* ref_ranks, double* rdm,
                                double* ranks, double* rho_out, void* workspace, int64_t workspace_bytes,
                                void* stream) {
  HBA_REQUIRE(E && ref_ranks && rho_out && N > 1 && Dm > 1, "hba_rdm_spearman: bad arguments");
  const int64_t P = (int64_t)N * (N - 1) / 2;
  HBA_REQUIRE(P > kSmallN, "hba_rdm_spearman: N=%d is served by hba_rdm_f64 + hba_rank_avg_f64 + hba_pearson_f64", N);
  HBA_REQUIRE(P < (1ll << 30), "hba_rdm_spearman: N too large");
  HBA_REQUIRE(workspace && workspace_bytes >= hba_rank_workspace_bytes(P) && ((uintptr_t)workspace & 255) == 0,
              "hba_rdm_spearman: workspace too small or not 256-byte aligned (need %lld bytes)",
              (long long)hba_rank_workspace_bytes(P));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const RankWorkspace w = rank_workspace_layout(workspace, P);
  launch_rdm(E, N, Dm, rdm, nullptr, w.k0, s);
  HBA_CHECK(check_launch("rdm_kernel"));
  return rank_large(nullptr, P, w, ranks, ref_ranks, rho_out, s);
}
