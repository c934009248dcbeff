// DoRA merge and its backward (reference: DoRALayer.weight, NEW:447-463, and the autograd mirror
// of those lines).  Bandwidth-bound: D is read once from HBM, every output written once.
//
//   V = D + scale * Bm @ A          D,V [in,out]; Bm [in,r]; A [r,out]
//   n_j = ||V[:,j]||_2 + eps        (eps added AFTER the sqrt, NEW:455)
//   Wt[i,j] = V[i,j] / n_j * m[j]   (the reference returns Wt^T as `.weight`)
//
// A CTA owns 8 consecutive output columns (one 32-byte sector per D row) and all `in` rows, so the
// column norm is a CTA-local reduction and D is read exactly once (single pass, V kept in
// registers).  The rank-r update costs in*out*r FMAs (33.5 M at 1024^2 x 32): negligible.
#include "common.cuh"

namespace hba {

constexpr int kDoraThreads = 256;
constexpr int kDoraCols = 8;
constexpr int kDoraMaxRows = 8;  // in_f <= 2048
constexpr int kDoraMaxRank = 64;

// v[k][j] for rows i = tid + 256 k; returns per-thread partial column sums of squares in ss[8]
__device__ __forceinline__ void dora_compute_v(const float* __restrict__ D,
                                               const float* __restrict__ Bm, const float (*sA)[kDoraCols],
                                               int in_f, int out_f, int r, float scale, int c0,
                                               float v[kDoraMaxRows][kDoraCols], float ss[kDoraCols]) {
#pragma unroll
  for (int j = 0; j < kDoraCols; ++j) ss[j] = 0.f;
#pragma unroll
  for (int k = 0; k < kDoraMaxRows; ++k) {
    const int i = threadIdx.x + kDoraThreads * k;
    if (i < in_f) {
      float acc[kDoraCols];
#pragma unroll
      for (int j = 0; j < kDoraCols; ++j) acc[j] = 0.f;
      const float* brow = Bm + (size_t)i * r;
      for (int kk = 0; kk < r; kk += 4) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(brow + kk));
#pragma unroll
        for (int j = 0; j < kDoraCols; ++j)
          acc[j] += b.x * sA[kk][j] + b.y * sA[kk + 1][j] + b.z * sA[kk + 2][j] + b.w * sA[kk + 3][j];
      }
      const float4 d0 = __ldg(reinterpret_cast<const float4*>(D + (size_t)i * out_f + c0));
      const float4 d1 = __ldg(reinterpret_cast<const float4*>(D + (size_t)i * out_f + c0 + 4));
      v[k][0] = d0.x + acc[0] * scale, v[k][1] = d0.y + acc[1] * scale;
      v[k][2] = d0.z + acc[2] * scale, v[k][3] = d0.w + acc[3] * scale;
      v[k][4] = d1.x + acc[4] * scale, v[k][5] = d1.y + acc[5] * scale;
      v[k][6] = d1.z + acc[6] * scale, v[k][7] = d1.w + acc[7] * scale;
#pragma unroll
      for (int j = 0; j < kDoraCols; ++j) ss[j] += v[k][j] * v[k][j];
    } else {
#pragma unroll
      for (int j = 0; j < kDoraCols; ++j) v[k][j] = 0.f;
    }
  }
}

// block-wide sums of 8 values, result broadcast to all threads through smem
__device__ __forceinline__ void block_sum8(float x[kDoraCols], float (*red)[kDoraCols]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < kDoraCols; ++j) x[j] = warp_sum(x[j]);
  __syncthreads();
  if (lane == 0)
#pragma unroll
    for (int j = 0; j < kDoraCols; ++j) red[warp][j] = x[j];
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kDoraCols; ++j) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kDoraThreads / 32; ++w) t += red[w][j];
    x[j] = t;
  }
}

__global__ void __launch_bounds__(kDoraThreads)
    dora_merge_fwd_kernel(const float* __restrict__ D, const float* __restrict__ A,
                          const float* __restrict__ Bm, const float* __restrict__ m, int in_f,
                          int out_f, int r, float scale, float eps, float* __restrict__ w_t_f32,
                          __nv_bfloat16* __restrict__ w_bf16, int64_t ld_w, int64_t w_lo_off,
                          __nv_bfloat16* __restrict__ wt_bf16, int64_t ld_wt, int64_t wt_lo_off,
                          float* __restrict__ norm_out) {
  __shared__ float sA[kDoraMaxRank][kDoraCols];
  __shared__ float red[kDoraThreads / 32][kDoraCols];
  const int c0 = blockIdx.x * kDoraCols;
  for (int i = threadIdx.x; i < r * kDoraCols; i += kDoraThreads)
    sA[i / kDoraCols][i % kDoraCols] = A[(size_t)(i / kDoraCols) * out_f + c0 + (i % kDoraCols)];
  __syncthreads();
  float v[kDoraMaxRows][kDoraCols], ss[kDoraCols];
  dora_compute_v(D, Bm, sA, in_f, out_f, r, scale, c0, v, ss);
  block_sum8(ss, red);
  float nrm[kDoraCols], mj[kDoraCols];
#pragma unroll
  for (int j = 0; j < kDoraCols; ++j) {
    nrm[j] = sqrtf(ss[j]) + eps;
    mj[j] = __ldg(m + c0 + j);
  }
  if (norm_out && threadIdx.x < kDoraCols) norm_out[c0 + threadIdx.x] = nrm[threadIdx.x];
#pragma unroll
  for (int k = 0; k < kDoraMaxRows; ++k) {
    const int i = threadIdx.x + kDoraThreads * k;
    if (i < in_f) {
      float w[kDoraCols];
#pragma unroll
      for (int j = 0; j < kDoraCols; ++j) w[j] = v[k][j] / nrm[j] * mj[j];
      if (w_t_f32) {
        float* o = w_t_f32 + (size_t)i * out_f + c0;
        *reinterpret_cast<float4*>(o) = make_float4(w[0], w[1], w[2], w[3]);
        *reinterpret_cast<float4*>(o + 4) = make_float4(w[4], w[5], w[6], w[7]);
      }
      if (wt_bf16) {
        __nv_bfloat16* o = wt_bf16 + (size_t)i * ld_wt + c0;
        *reinterpret_cast<uint4*>(o) = make_uint4(pack_bf16x2(w[0], w[1]), pack_bf16x2(w[2], w[3]),
                                                  pack_bf16x2(w[4], w[5]), pack_bf16x2(w[6], w[7]));
        if (wt_lo_off > 0) {
          float l[kDoraCols];
#pragma unroll
          for (int j = 0; j < kDoraCols; ++j) l[j] = w[j] - __bfloat162float(__float2bfloat16_rn(w[j]));
          *reinterpret_cast<uint4*>(o + wt_lo_off) =
              make_uint4(pack_bf16x2(l[0], l[1]), pack_bf16x2(l[2], l[3]), pack_bf16x2(l[4], l[5]),
                         pack_bf16x2(l[6], l[7]));
        }
      }
      if (w_bf16) {
#pragma unroll
        for (int j = 0; j < kDoraCols; ++j) {
          __nv_bfloat16 h, l;
          split_bf16(w[j], h, l);
          w_bf16[(size_t)(c0 + j) * ld_w + i] = h;
          if (w_lo_off > 0) w_bf16[(size_t)(c0 + j) * ld_w + w_lo_off + i] = l;
        }
      }
    }
  }
}

// backward, phase 1 (column-owning CTAs): dm, dA and dV (written to the workspace)
__global__ void __launch_bounds__(kDoraThreads)
    dora_merge_bwd_cols_kernel(const float* __restrict__ G, int64_t ld_g,
                               const float* __restrict__ D, const float* __restrict__ A,
                               const float* __restrict__ Bm, const float* __restrict__ m, int in_f,
                               int out_f, int r, float scale, float eps, float* __restrict__ dm,
                               float* __restrict__ dA, float* __restrict__ dV) {
  __shared__ float sA[kDoraMaxRank][kDoraCols];
  __shared__ float red[kDoraThreads / 32][kDoraCols];
  extern __shared__ __align__(16) float sDV[];  // [in_f][8]
  const int c0 = blockIdx.x * kDoraCols;
  for (int i = threadIdx.x; i < r * kDoraCols; i += kDoraThreads)
    sA[i / kDoraCols][i % kDoraCols] = A[(size_t)(i / kDoraCols) * out_f + c0 + (i % kDoraCols)];
  __syncthreads();
  float v[kDoraMaxRows][kDoraCols], ss[kDoraCols];
  dora_compute_v(D, Bm, sA, in_f, out_f, r, scale, c0, v, ss);
  block_sum8(ss, red);
  float g[kDoraMaxRows][kDoraCols], c[kDoraCols];
#pragma unroll
  for (int j = 0; j < kDoraCols; ++j) c[j] = 0.f;
#pragma unroll
  for (int k = 0; k < kDoraMaxRows; ++k) {
    const int i = threadIdx.x + kDoraThreads * k;
#pragma unroll
    for (int j = 0; j < kDoraCols; ++j) {
      g[k][j] = (i < in_f) ? __ldg(G + (size_t)(c0 + j) * ld_g + i) : 0.f;
      c[j] += g[k][j] * v[k][j];
    }
  }
  block_sum8(c, red);
  float coef[kDoraCols], back[kDoraCols];
#pragma unroll
  for (int j = 0; j < kDoraCols; ++j) {
    const float vn = sqrtf(ss[j]);
    const float n = vn + eps;
    const float mj = __ldg(m + c0 + j);
    coef[j] = mj / n;
    back[j] = (vn > 0.f) ? c[j] / (n * vn) : 0.f;
    if (threadIdx.x == j) dm[c0 + j] = c[j] / n;
  }
#pragma unroll
  for (int k = 0; k < kDoraMaxRows; ++k) {
    const int i = threadIdx.x + kDoraThreads * k;
    if (i < in_f) {
      float dv[kDoraCols];
#pragma unroll
      for (int j = 0; j < kDoraCols; ++j) dv[j] = coef[j] * (g[k][j] - v[k][j] * back[j]);
      *reinterpret_cast<float4*>(sDV + (size_t)i * kDoraCols) = make_float4(dv[0], dv[1], dv[2], dv[3]);
      *reinterpret_cast<float4*>(sDV + (size_t)i * kDoraCols + 4) = make_float4(dv[4], dv[5], dv[6], dv[7]);
      float* o = dV + (size_t)i * out_f + c0;
      *reinterpret_cast<float4*>(o) = make_float4(dv[0], dv[1], dv[2], dv[3]);
      *reinterpret_cast<float4*>(o + 4) = make_float4(dv[4], dv[5], dv[6], dv[7]);
    }
  }
  __syncthreads();
  // dA[k, c0 + j] = scale * sum_i Bm[i,k] dV[i,j].  Lane = rank index k (two per lane when r > 32), the
  // 8 warps split the rows: every Bm row (one 128-byte line at r = 32) is read exactly once, coalesced,
  // 16 rows in flight per warp; dV[i, j] is a shared-memory broadcast.  Cross-warp sum through smem.
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float accA[2][kDoraCols];
#pragma unroll
  for (int h2 = 0; h2 < 2; ++h2)
#pragma unroll
    for (int j = 0; j < kDoraCols; ++j) accA[h2][j] = 0.f;
  const int rows_per_warp = (in_f + 7) / 8;
  const int i_begin = warp * rows_per_warp, i_end = min(in_f, i_begin + rows_per_warp);
  for (int i0 = i_begin; i0 < i_end; i0 += 16) {
    float b0[16], b1[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const int i = i0 + u;
      b0[u] = (i < i_end && lane < r) ? __ldg(Bm + (size_t)i * r + lane) : 0.f;
      b1[u] = (i < i_end && lane + 32 < r) ? __ldg(Bm + (size_t)i * r + lane + 32) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const int i = min(i0 + u, in_f - 1);
      const float4 d0 = *reinterpret_cast<const float4*>(sDV + (size_t)i * kDoraCols);
      const float4 d1 = *reinterpret_cast<const float4*>(sDV + (size_t)i * kDoraCols + 4);
      const float dv[kDoraCols] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
      for (int j = 0; j < kDoraCols; ++j) {
        accA[0][j] += b0[u] * dv[j];
        accA[1][j] += b1[u] * dv[j];
      }
    }
  }
  __syncthreads();  // every warp is done reading sDV: reuse it for the per-warp partial sums
  float* part = sDV;  // [8 warps][64 k][8 j] floats = 16 KB (the launcher reserves at least that)
#pragma unroll
  for (int h2 = 0; h2 < 2; ++h2)
#pragma unroll
    for (int j = 0; j < kDoraCols; ++j)
      part[((size_t)warp * 64 + lane + 32 * h2) * kDoraCols + j] = accA[h2][j];
  __syncthreads();
  for (int t = threadIdx.x; t < r * kDoraCols; t += kDoraThreads) {
    const int k = t / kDoraCols, j = t % kDoraCols;
    float acc = 0.f;
#pragma unroll
    for (int w = 0; w < kDoraThreads / 32; ++w) acc += part[((size_t)w * 64 + k) * kDoraCols + j];
    dA[(size_t)k * out_f + c0 + j] = scale * acc;
  }
}

// backward, phase 2 (row-owning warps): dB[i,k] = scale * sum_j dV[i,j] A[k,j].
// The CTA stages 32 rank rows of A (all out_f columns, <= 2048) in shared memory once; a warp owns
// one row i, its lanes split the columns (coalesced reads of dV, 32 loads in flight), every lane keeps
// 32 partial sums (one per rank index) and the warp reduces them with shuffles at the end.
__global__ void __launch_bounds__(256)
    dora_merge_bwd_rows_kernel(const float* __restrict__ dV, const float* __restrict__ A, int in_f,
                               int out_f, int r, float scale, float* __restrict__ dB) {
  extern __shared__ __align__(16) float sAr[];  // [32][out_f + 1]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + warp;
  const int pitch = out_f + 1;
  for (int k0 = 0; k0 < r; k0 += 32) {
    __syncthreads();
    for (int t = threadIdx.x; t < 32 * (out_f / 4); t += 256) {
      const int k = t / (out_f / 4), j4 = (t % (out_f / 4)) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (k0 + k < r) v = __ldg(reinterpret_cast<const float4*>(A + (size_t)(k0 + k) * out_f + j4));
      float* dst = sAr + (size_t)k * pitch + j4;
      dst[0] = v.x, dst[1] = v.y, dst[2] = v.z, dst[3] = v.w;
    }
    __syncthreads();
    if (i < in_f) {
      float acc[32];
#pragma unroll
      for (int k = 0; k < 32; ++k) acc[k] = 0.f;
      for (int c0 = 0; c0 < out_f; c0 += 256) {
        float dv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int j = c0 + lane + 32 * u;
          dv[u] = (j < out_f) ? __ldg(dV + (size_t)i * out_f + j) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int j = min(c0 + lane + 32 * u, out_f - 1);
#pragma unroll
          for (int k = 0; k < 32; ++k) acc[k] += dv[u] * sAr[(size_t)k * pitch + j];
        }
      }
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const float t = warp_sum(acc[k]);
        if (lane == k && k0 + k < r) dB[(size_t)i * r + k0 + k] = scale * t;
      }
    }
  }
}

// =============================================================================================
// Cluster form (in_f <= 1024, in_f % 8 == 0, out_f % 32 == 0, r <= 32): what the step runs.
// A CTA owns a 128-row x 32-column tile of D (rows of one 128-byte line each: every global access of the
// kernel is a full line), the <= 8 CTAs that share a column block form one thread-block cluster and exchange
// their column partial sums (||V_j||^2, <G_j, V_j>, dA) through distributed shared memory in a fixed order, so
// results are deterministic and D / G are read exactly once.  Grid = (out_f / 32) x ceil(in_f / 128) CTAs:
// 256 at 1024^2, i.e. one wave at <= 2 CTAs per SM instead of 128 CTAs with 4 KB-strided 32-byte accesses.
constexpr int kTR = 128;     // rows per CTA
constexpr int kTC = 32;      // columns per CTA
constexpr int kPitch = 33;   // shared-memory row pitch (floats): conflict-free row- and column-wise
constexpr int kRankMax = 32;

__device__ __forceinline__ float ld_dsmem_f32(const float* p, uint32_t rank) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(mapa_u32(p, rank)) : "memory");
  return v;
}

// A tile [r][32] and B tile [128][r] -> shared memory (pitch 33); rows beyond in_f are zero
__device__ __forceinline__ void dora_stage_ab(const float* __restrict__ A, const float* __restrict__ Bm, int in_f,
                                              int out_f, int r, int c0, int i0, float (*sA)[kPitch],
                                              float (*sB)[kPitch]) {
  for (int idx = threadIdx.x; idx < r * kTC; idx += kDoraThreads)
    sA[idx / kTC][idx % kTC] = __ldg(A + (size_t)(idx / kTC) * out_f + c0 + (idx % kTC));
  for (int idx = threadIdx.x; idx < kTR * r; idx += kDoraThreads) {
    const int i = idx / r, k = idx % r;
    sB[i][k] = (i0 + i < in_f) ? __ldg(Bm + (size_t)(i0 + i) * r + k) : 0.f;
  }
}

// v[u][e] = D + scale * (B A) for rows r0 + 32 u, columns 4 cg + e of the tile (0 beyond in_f)
__device__ __forceinline__ void dora_tile_v(const float* __restrict__ D, int in_f, int out_f, int r, float scale,
                                            int c0, int i0, const float (*sA)[kPitch], const float (*sB)[kPitch],
                                            float v[4][4]) {
  const int cg = threadIdx.x & 7, r0 = threadIdx.x >> 3;
  float4 d[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int i = i0 + r0 + 32 * u;
    d[u] = (i < in_f) ? __ldg(reinterpret_cast<const float4*>(D + (size_t)i * out_f + c0 + 4 * cg))
                      : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float acc[4][4];
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int e = 0; e < 4; ++e) acc[u][e] = 0.f;
  for (int kk = 0; kk < r; ++kk) {
    float a[4], b[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) a[e] = sA[kk][4 * cg + e];
#pragma unroll
    for (int u = 0; u < 4; ++u) b[u] = sB[r0 + 32 * u][kk];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[u][e] = fmaf(b[u], a[e], acc[u][e]);
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const bool ok = i0 + r0 + 32 * u < in_f;
    v[u][0] = ok ? d[u].x + acc[u][0] * scale : 0.f;
    v[u][1] = ok ? d[u].y + acc[u][1] * scale : 0.f;
    v[u][2] = ok ? d[u].z + acc[u][2] * scale : 0.f;
    v[u][3] = ok ? d[u].w + acc[u][3] * scale : 0.f;
  }
}

// x[e] (one value per column 4 cg + e of this thread) -> sums over the CTA's 128 rows in out[0..31]
// (fixed order: lanes by xor-shuffle, then warps 0..7); `red` = [8][32] scratch.  Ends with __syncthreads.
__device__ __forceinline__ void dora_colsum_cta(float x[4], float (*red)[kTC], float* out) {
  const int cg = threadIdx.x & 7, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    x[e] += __shfl_xor_sync(0xffffffffu, x[e], 8);
    x[e] += __shfl_xor_sync(0xffffffffu, x[e], 16);
  }
  if (lane < 8) {
#pragma unroll
    for (int e = 0; e < 4; ++e) red[warp][4 * cg + e] = x[e];
  }
  __syncthreads();
  if (threadIdx.x < kTC) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kDoraThreads / 32; ++w) t += red[w][threadIdx.x];
    out[threadIdx.x] = t;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kDoraThreads)
    dora_fwd_cluster_kernel(const float* __restrict__ D, const float* __restrict__ A, const float* __restrict__ Bm,
                            const float* __restrict__ m, int in_f, int out_f, int r, float scale, float eps,
                            float* __restrict__ w_t_f32, __nv_bfloat16* __restrict__ w_bf16, int64_t ld_w,
                            int64_t w_lo_off, __nv_bfloat16* __restrict__ wt_bf16, int64_t ld_wt, int64_t wt_lo_off,
                            float* __restrict__ norm_out) {
  __shared__ float sA[kRankMax][kPitch];
  __shared__ float sB[kTR][kPitch];
  __shared__ float red[kDoraThreads / 32][kTC];
  __shared__ float s_part[kTC];   // this CTA's column sums of squares (read by the whole cluster)
  __shared__ float s_tot[kTC];
  __shared__ __align__(16) __nv_bfloat16 s_hi[kTC][kTR + 8];   // transposed staging of the W operand
  __shared__ __align__(16) __nv_bfloat16 s_lo[kTC][kTR + 8];
  const int c0 = blockIdx.x * kTC, rank = blockIdx.y, cs = gridDim.y, i0 = rank * kTR;
  const int cg = threadIdx.x & 7, r0 = threadIdx.x >> 3;
  dora_stage_ab(A, Bm, in_f, out_f, r, c0, i0, sA, sB);
  __syncthreads();
  float v[4][4];
  dora_tile_v(D, in_f, out_f, r, scale, c0, i0, sA, sB, v);
  float ss[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) ss[e] = v[0][e] * v[0][e] + v[1][e] * v[1][e] + v[2][e] * v[2][e] + v[3][e] * v[3][e];
  dora_colsum_cta(ss, red, s_part);
  cluster_sync_all();
  if (threadIdx.x < kTC) {
    float t = 0.f;
    for (int q = 0; q < cs; ++q) t += ld_dsmem_f32(&s_part[threadIdx.x], q);
    s_tot[threadIdx.x] = t;
  }
  cluster_sync_all();   // every remote read is done (no CTA may leave earlier) and s_tot is visible
  float nrm[4], mj[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    nrm[e] = sqrtf(s_tot[4 * cg + e]) + eps;
    mj[e] = __ldg(m + c0 + 4 * cg + e);
  }
  if (norm_out && rank == 0 && threadIdx.x < kTC) norm_out[c0 + threadIdx.x] = sqrtf(s_tot[threadIdx.x]) + eps;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int il = r0 + 32 * u, i = i0 + il;
    float w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) w[e] = v[u][e] / nrm[e] * mj[e];
    if (w_bf16) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        __nv_bfloat16 h, l;
        split_bf16(w[e], h, l);
        s_hi[4 * cg + e][il] = h;
        s_lo[4 * cg + e][il] = l;
      }
    }
    if (i >= in_f) continue;
    if (w_t_f32) *reinterpret_cast<float4*>(w_t_f32 + (size_t)i * out_f + c0 + 4 * cg) = make_float4(w[0], w[1], w[2], w[3]);
    if (wt_bf16) {
      __nv_bfloat16* o = wt_bf16 + (size_t)i * ld_wt + c0 + 4 * cg;
      *reinterpret_cast<uint2*>(o) = make_uint2(pack_bf16x2(w[0], w[1]), pack_bf16x2(w[2], w[3]));
      if (wt_lo_off > 0) {
        float l[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) l[e] = w[e] - __bfloat162float(__float2bfloat16_rn(w[e]));
        *reinterpret_cast<uint2*>(o + wt_lo_off) = make_uint2(pack_bf16x2(l[0], l[1]), pack_bf16x2(l[2], l[3]));
      }
    }
  }
  if (w_bf16) {
    __syncthreads();
    // W [out, in]: column j of the tile is a run of 128 consecutive bf16 of row c0 + j; thread = (column, 16 rows)
    const int col = threadIdx.x >> 3, seg = (threadIdx.x & 7) * 16;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int il = seg + 8 * h;
      if (i0 + il < in_f) {   // in_f % 8 == 0: whole groups of 8
        __nv_bfloat16* o = w_bf16 + (size_t)(c0 + col) * ld_w + i0 + il;
        *reinterpret_cast<uint4*>(o) = *reinterpret_cast<const uint4*>(&s_hi[col][il]);
        if (w_lo_off > 0) *reinterpret_cast<uint4*>(o + w_lo_off) = *reinterpret_cast<const uint4*>(&s_lo[col][il]);
      }
    }
  }
}

// Backward: dm, dA through the cluster; dB as per-column-block partial sums dBp[cb][in][r] (reduced in a fixed order
// by dora_db_reduce_kernel).  G = dL/dW in [out, ld_g] layout.
struct DoraBwdSmem {
  float sA[kRankMax][kPitch];
  float sB[kTR][kPitch];
  float sGV[kTR * kPitch];          // G tile as [32][129] (transposed read), then dV as [128][33], then dA scratch
  float red[kDoraThreads / 32][kTC];
  float s_part[2][kTC];             // column partials of this CTA: ||V||^2 and <G, V>
  float s_tot[2][kTC];
  float s_pa[kRankMax][kTC];        // this CTA's partial dA (read by the whole cluster)
};

__global__ void __launch_bounds__(kDoraThreads)
    dora_bwd_cluster_kernel(const float* __restrict__ G, int64_t ld_g, const float* __restrict__ D,
                            const float* __restrict__ A, const float* __restrict__ Bm, const float* __restrict__ m,
                            int in_f, int out_f, int r, float scale, float eps, float* __restrict__ dm,
                            float* __restrict__ dA, float* __restrict__ dBp) {
  extern __shared__ __align__(16) uint8_t dora_smem[];
  DoraBwdSmem& S = *reinterpret_cast<DoraBwdSmem*>(dora_smem);
  const int c0 = blockIdx.x * kTC, rank = blockIdx.y, cs = gridDim.y, i0 = rank * kTR;
  const int cg = threadIdx.x & 7, r0 = threadIdx.x >> 3;
  dora_stage_ab(A, Bm, in_f, out_f, r, c0, i0, S.sA, S.sB);
  // G tile: row c0 + j of G holds the 128 values G[j, i0 .. i0 + 127] contiguously
  constexpr int kGP = kTR + 1;
  for (int idx = threadIdx.x; idx < kTC * kTR; idx += kDoraThreads) {
    const int j = idx / kTR, i = idx % kTR;
    S.sGV[j * kGP + i] = (i0 + i < in_f) ? __ldg(G + (size_t)(c0 + j) * ld_g + i0 + i) : 0.f;
  }
  __syncthreads();
  float v[4][4], g[4][4];
  dora_tile_v(D, in_f, out_f, r, scale, c0, i0, S.sA, S.sB, v);
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int e = 0; e < 4; ++e) g[u][e] = S.sGV[(4 * cg + e) * kGP + r0 + 32 * u];
  float ss[4], cc[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    ss[e] = v[0][e] * v[0][e] + v[1][e] * v[1][e] + v[2][e] * v[2][e] + v[3][e] * v[3][e];
    cc[e] = g[0][e] * v[0][e] + g[1][e] * v[1][e] + g[2][e] * v[2][e] + g[3][e] * v[3][e];
  }
  dora_colsum_cta(ss, S.red, S.s_part[0]);
  dora_colsum_cta(cc, S.red, S.s_part[1]);
  cluster_sync_all();
  if (threadIdx.x < 2 * kTC) {
    const int which = threadIdx.x / kTC, j = threadIdx.x % kTC;
    float t = 0.f;
    for (int q = 0; q < cs; ++q) t += ld_dsmem_f32(&S.s_part[which][j], q);
    S.s_tot[which][j] = t;
  }
  cluster_sync_all();
  float coef[4], back[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float vn = sqrtf(S.s_tot[0][4 * cg + e]);
    const float n = vn + eps;
    const float c = S.s_tot[1][4 * cg + e];
    coef[e] = __ldg(m + c0 + 4 * cg + e) / n;
    back[e] = (vn > 0.f) ? c / (n * vn) : 0.f;
  }
  if (rank == 0 && threadIdx.x < kTC) {
    const float vn = sqrtf(S.s_tot[0][threadIdx.x]);
    dm[c0 + threadIdx.x] = S.s_tot[1][threadIdx.x] / (vn + eps);
  }
  // dV tile -> shared memory [128][33] (over the G tile: every thread has taken its G values into registers)
  __syncthreads();
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int e = 0; e < 4; ++e)
      S.sGV[(r0 + 32 * u) * kPitch + 4 * cg + e] = coef[e] * (g[u][e] - v[u][e] * back[e]);
  __syncthreads();
  // ---- dB partial of this column block: dBp[cb][i][k] = sum_j dV[i,j] A[k,j]; thread = 4 rows x 4 rank indices
  {
    const int kg = threadIdx.x & 7, rg = threadIdx.x >> 3;
    float acc[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[u][q] = 0.f;
    if (4 * kg < r) {
#pragma unroll 8
      for (int j = 0; j < kTC; ++j) {
        float dv[4], a[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) dv[u] = S.sGV[(rg + 32 * u) * kPitch + j];
#pragma unroll
        for (int q = 0; q < 4; ++q) a[q] = S.sA[4 * kg + q][j];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[u][q] = fmaf(dv[u], a[q], acc[u][q]);
      }
      float* base = dBp + (size_t)blockIdx.x * in_f * r;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + rg + 32 * u;
        if (i < in_f)
          *reinterpret_cast<float4*>(base + (size_t)i * r + 4 * kg) = make_float4(acc[u][0], acc[u][1], acc[u][2], acc[u][3]);
      }
    }
  }
  // ---- dA partial of this CTA's rows: sum_i B[i,k] dV[i,j]; thread = 4 rank indices x 4 columns x a quarter of
  // the rows, the four row quarters are added in a fixed order through shared memory
  float pa[4][4];
  {
    const int jg = threadIdx.x & 7, kq = (threadIdx.x >> 3) & 7, ih = threadIdx.x >> 6;
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int e = 0; e < 4; ++e) pa[q][e] = 0.f;
#pragma unroll 4
    for (int i = 32 * ih; i < 32 * ih + 32; ++i) {
      float b[4], dv[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) b[q] = S.sB[i][4 * kq + q];   // (columns >= r of sB are never written: guarded below)
#pragma unroll
      for (int e = 0; e < 4; ++e) dv[e] = S.sGV[i * kPitch + 4 * jg + e];
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int e = 0; e < 4; ++e) pa[q][e] = fmaf(b[q], dv[e], pa[q][e]);
    }
  }
  __syncthreads();   // dV is no longer needed: its storage becomes the [4 quarters][32 k][32 j] scratch
  {
    const int jg = threadIdx.x & 7, kq = (threadIdx.x >> 3) & 7, ih = threadIdx.x >> 6;
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int e = 0; e < 4; ++e) S.sGV[(ih * kRankMax + 4 * kq + q) * kTC + 4 * jg + e] = pa[q][e];
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < kRankMax * kTC; idx += kDoraThreads) {
    float t = 0.f;
#pragma unroll
    for (int ih = 0; ih < 4; ++ih) t += S.sGV[ih * kRankMax * kTC + idx];
    S.s_pa[idx / kTC][idx % kTC] = t;
  }
  cluster_sync_all();
  // dA[k, c0 + j] = scale * sum over the cluster's CTAs (rank order); rank q writes the rows k = q, q + cs, ...
  for (int idx = threadIdx.x; idx < r * kTC; idx += kDoraThreads) {
    const int k = idx / kTC, j = idx % kTC;
    if (k % cs != rank) continue;
    float t = 0.f;
    for (int q = 0; q < cs; ++q) t += ld_dsmem_f32(&S.s_pa[k][j], q);
    dA[(size_t)k * out_f + c0 + j] = scale * t;
  }
  cluster_sync_all();   // no CTA leaves while its partials are still being read
}

// dB[i, k] = scale * sum_cb dBp[cb][i][k]  (fixed order)
__global__ void __launch_bounds__(256)
    dora_db_reduce_kernel(const float* __restrict__ dBp, int ncb, int64_t n4, float scale, float* __restrict__ dB) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n4) return;
  float4 acc = __ldg(reinterpret_cast<const float4*>(dBp) + i);
  for (int cb = 1; cb < ncb; ++cb) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(dBp) + (size_t)cb * n4 + i);
    acc.x += t.x, acc.y += t.y, acc.z += t.z, acc.w += t.w;
  }
  reinterpret_cast<float4*>(dB)[i] = make_float4(scale * acc.x, scale * acc.y, scale * acc.z, scale * acc.w);
}

static bool dora_cluster_ok(int in_f, int out_f, int r) {
  return in_f <= 8 * kTR && in_f % 8 == 0 && out_f % kTC == 0 && r <= kRankMax && r % 4 == 0;
}

template <typename Kernel, typename... Args>
static int launch_dora_cluster(Kernel kernel, const char* name, int out_f, int in_f, size_t smem, cudaStream_t s,
                               Args... args) {
  cudaLaunchConfig_t cfg = {};
  const unsigned cs = (unsigned)((in_f + kTR - 1) / kTR);
  cfg.gridDim = dim3((unsigned)(out_f / kTC), cs, 1);
  cfg.blockDim = dim3(kDoraThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1;
  attr[0].val.clusterDim.y = cs;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, args...);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("%s launch: %s", name, cudaGetErrorString(e));
    return HBA_ERR_CUDA;
  }
  return check_launch(name);
}

}  // namespace hba

using namespace hba;

static int dora_check(const char* who, int in_f, int out_f, int r) {
  HBA_REQUIRE(in_f > 0 && in_f <= kDoraThreads * kDoraMaxRows, "%s: in_features=%d unsupported (max %d)", who, in_f, kDoraThreads * kDoraMaxRows);
  HBA_REQUIRE(out_f > 0 && out_f % kDoraCols == 0, "%s: out_features=%d must be a multiple of %d", who, out_f, kDoraCols);
  HBA_REQUIRE(r > 0 && r <= kDoraMaxRank && r % 4 == 0, "%s: rank=%d must be a multiple of 4 and <= %d", who, r, kDoraMaxRank);
  return HBA_OK;
}

extern "C" int hba_dora_merge_fwd(const float* D, const float* A, const float* Bm, const float* m,
                                  int32_t in_f, int32_t out_f, int32_t r, float scale, float eps,
                                  float* w_t_f32, void* w_bf16, int64_t ld_w, int64_t w_lo_off,
                                  void* wt_bf16, int64_t ld_wt, int64_t wt_lo_off, float* norm_out,
                                  void* stream) {
  HBA_REQUIRE(D && A && Bm && m, "hba_dora_merge_fwd: null input");
  HBA_REQUIRE(w_t_f32 || w_bf16 || wt_bf16, "hba_dora_merge_fwd: no output requested");
  HBA_CHECK(dora_check("hba_dora_merge_fwd", in_f, out_f, r));
  HBA_REQUIRE(!wt_bf16 || (ld_wt % 8 == 0 && wt_lo_off % 8 == 0 && ((uintptr_t)wt_bf16 & 15) == 0), "hba_dora_merge_fwd: wt_bf16 alignment");
  if (dora_cluster_ok(in_f, out_f, r) && (!w_bf16 || (ld_w % 8 == 0 && w_lo_off % 8 == 0 && ((uintptr_t)w_bf16 & 15) == 0)) &&
      (!w_t_f32 || ((uintptr_t)w_t_f32 & 15) == 0) && ((uintptr_t)D & 15) == 0)
    return launch_dora_cluster(dora_fwd_cluster_kernel, "dora_fwd_cluster_kernel", out_f, in_f, 0,
                               static_cast<cudaStream_t>(stream), D, A, Bm, m, (int)in_f, (int)out_f, (int)r, scale,
                               eps, w_t_f32, static_cast<__nv_bfloat16*>(w_bf16), ld_w, w_lo_off,
                               static_cast<__nv_bfloat16*>(wt_bf16), ld_wt, wt_lo_off, norm_out);
  dora_merge_fwd_kernel<<<out_f / kDoraCols, kDoraThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      D, A, Bm, m, in_f, out_f, r, scale, eps, w_t_f32, static_cast<__nv_bfloat16*>(w_bf16), ld_w,
      w_lo_off, static_cast<__nv_bfloat16*>(wt_bf16), ld_wt, wt_lo_off, norm_out);
  return check_launch("dora_merge_fwd_kernel");
}

extern "C" int hba_dora_merge_bwd(const float* G, int64_t ld_g, const float* D, const float* A,
                                  const float* Bm, const float* m, int32_t in_f, int32_t out_f,
                                  int32_t r, float scale, float eps, float* dm, float* dA, float* dB,
                                  float* workspace, void* stream) {
  HBA_REQUIRE(G && D && A && Bm && m && dm && dA && dB && workspace, "hba_dora_merge_bwd: null pointer");
  HBA_CHECK(dora_check("hba_dora_merge_bwd", in_f, out_f, r));
  HBA_REQUIRE(out_f <= 1792, "hba_dora_merge_bwd: out_features=%d exceeds the shared-memory staging (max 1792)", out_f);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dora_cluster_ok(in_f, out_f, r) && ((uintptr_t)D & 15) == 0 && ((uintptr_t)workspace & 15) == 0 &&
      ((uintptr_t)dB & 15) == 0) {
    // workspace [out_f / 32][in_f][r] floats <= in_f * out_f (r <= 32)
    static SmemAttr attr;
    HBA_CHECK(ensure_dyn_smem(dora_bwd_cluster_kernel, sizeof(DoraBwdSmem), attr, "dora_bwd_cluster_kernel"));
    HBA_CHECK(launch_dora_cluster(dora_bwd_cluster_kernel, "dora_bwd_cluster_kernel", out_f, in_f, sizeof(DoraBwdSmem),
                                  s, G, ld_g, D, A, Bm, m, (int)in_f, (int)out_f, (int)r, scale, eps, dm, dA,
                                  workspace));
    const int64_t n4 = (int64_t)in_f * r / 4;
    dora_db_reduce_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, s>>>(workspace, out_f / kTC, n4, scale, dB);
    return check_launch("dora_db_reduce_kernel");
  }
  // [in_f][8] dV tile, later reused for the [8 warps][64][8] partial sums of dA
  const size_t smem = (size_t)(in_f > 512 ? in_f : 512) * kDoraCols * sizeof(float);
  static SmemAttr attr_cols;
  if (smem > 48 * 1024 - 4096)
    HBA_CHECK(ensure_dyn_smem(dora_merge_bwd_cols_kernel, smem, attr_cols, "dora_merge_bwd_cols_kernel"));
  dora_merge_bwd_cols_kernel<<<out_f / kDoraCols, kDoraThreads, smem, s>>>(
      G, ld_g, D, A, Bm, m, in_f, out_f, r, scale, eps, dm, dA, workspace);
  HBA_CHECK(check_launch("dora_merge_bwd_cols_kernel"));
  const size_t smem_rows = (size_t)32 * (out_f + 1) * sizeof(float);
  static SmemAttr attr_rows;
  HBA_CHECK(ensure_dyn_smem(dora_merge_bwd_rows_kernel, smem_rows, attr_rows, "dora_merge_bwd_rows_kernel"));
  dora_merge_bwd_rows_kernel<<<(in_f + 7) / 8, 256, smem_rows, s>>>(workspace, A, in_f, out_f, r, scale, dB);
  return check_launch("dora_merge_bwd_rows_kernel");
}
