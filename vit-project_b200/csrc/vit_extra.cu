// Kernels that only the fully-trained ViT-B/16 data-parallel baseline needs (reference VIT:125-165,
// every parameter trainable): column sums (bias gradients), LayerNorm parameter gradients, and the
// full softmax-attention backward (dQ, dK, dV for every row).
#include "common.cuh"

namespace hba {

template <typename T>
__device__ __forceinline__ float to_f(T v);
template <>
__device__ __forceinline__ float to_f<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T>
__device__ __forceinline__ T from_f(float v);
template <>
__device__ __forceinline__ float from_f<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// ------------------------------------------------------------------------------------------
// column sums: partial[chunk, c] = sum over the chunk's rows of x[r, c] (optionally x * xhat terms
// for LayerNorm parameter gradients); deterministic two-stage reduction.
constexpr int kCsChunks = 128;

template <typename T>
__global__ void __launch_bounds__(256)
    colsum_partial_kernel(const T* __restrict__ x, int64_t rows, int cols, int64_t ld,
                          float* __restrict__ partial) {
  __shared__ float red[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int64_t per = (rows + kCsChunks - 1) / kCsChunks;
  const int64_t r0 = (int64_t)blockIdx.y * per, r1 = min(r0 + per, rows);
  float s = 0.f;
  if (c < cols)
    for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) s += to_f(x[r * ld + c]);
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && c < cols) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
    partial[(size_t)blockIdx.y * cols + c] = t;
  }
}

// LayerNorm parameter gradients: dgamma[c] = sum_r dy[r,c] * xhat[r,c], dbeta[c] = sum_r dy[r,c]
__global__ void __launch_bounds__(256)
    ln_param_partial_kernel(const float* __restrict__ dy, int64_t ld_dy, const float* __restrict__ x,
                            int64_t ldx, int64_t row_step, const float* __restrict__ stats,
                            int64_t rows, int cols, float* __restrict__ partial) {
  __shared__ float red[2][8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int64_t per = (rows + kCsChunks - 1) / kCsChunks;
  const int64_t r0 = (int64_t)blockIdx.y * per, r1 = min(r0 + per, rows);
  float sg = 0.f, sb = 0.f;
  if (c < cols)
    for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) {
      const float mean = stats[2 * r], rstd = stats[2 * r + 1];
      const float d = dy[r * ld_dy + c];
      sg += d * (x[r * row_step * ldx + c] - mean) * rstd;
      sb += d;
    }
  red[0][threadIdx.y][threadIdx.x] = sg;
  red[1][threadIdx.y][threadIdx.x] = sb;
  __syncthreads();
  if (threadIdx.y == 0 && c < cols) {
    float tg = 0.f, tb = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) tg += red[0][k][threadIdx.x], tb += red[1][k][threadIdx.x];
    partial[(size_t)blockIdx.y * 2 * cols + c] = tg;
    partial[(size_t)blockIdx.y * 2 * cols + cols + c] = tb;
  }
}

__global__ void colsum_final_kernel(const float* __restrict__ partial, int width,
                                    float* __restrict__ out, int accumulate) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= width) return;
  float t = 0.f;
  for (int k = 0; k < kCsChunks; ++k) t += partial[(size_t)k * width + c];
  out[c] = accumulate ? out[c] + t : t;
}

// per-row LayerNorm statistics (mean, rstd), one warp per row
__global__ void __launch_bounds__(256)
    ln_stats_kernel(const float* __restrict__ x, int64_t rows, int cols, int64_t ldx, int64_t row_step,
                    float eps, float* __restrict__ stats) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + row * row_step * ldx;
  float s = 0.f;
  for (int c = lane * 4; c < cols; c += 128) {
    const float4 v = *reinterpret_cast<const float4*>(xr + c);
    s += (v.x + v.y) + (v.z + v.w);
  }
  const float mean = warp_sum(s) / cols;
  float sq = 0.f;
  for (int c = lane * 4; c < cols; c += 128) {
    const float4 v = *reinterpret_cast<const float4*>(xr + c);
    const float a = v.x - mean, b = v.y - mean, cc = v.z - mean, d = v.w - mean;
    sq += (a * a + b * b) + (cc * cc + d * d);
  }
  const float rstd = rsqrtf(warp_sum(sq) / cols + eps);
  if (lane == 0) stats[2 * row] = mean, stats[2 * row + 1] = rstd;
}

// ------------------------------------------------------------------------------------------
// Fused LayerNorm backward of the fully-trained ViT (replaces five passes over the [rows, cols]
// gradients: statistics, dx, dgamma / dbeta partials, the bf16 copy of dx that feeds the next GEMMs and
// the column sums of dx = the bias gradient of the Linear in front of the LayerNorm's input):
//   dx (+)= rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma
//   part[block][0:cols] = sum dy * xhat, [cols:2cols] = sum dy, [2cols:3cols] = sum dx (after +=)
// One warp per row, rows cyclic over all warps of the grid; every lane keeps its NVEC*4 columns of the
// three column sums in registers over all its rows (deterministic: fixed row -> warp assignment,
// fixed reduction order).  HBM traffic: read dy, x (, dx) + write dx fp32 (, bf16) - one pass.
template <int NVEC>
__global__ void __launch_bounds__(256)
    layernorm_bwd_fused_kernel(const float* __restrict__ dy, int64_t ld_dy, const float* __restrict__ x,
                               int64_t rows, int64_t ldx, const float* __restrict__ gamma, float eps,
                               float* dx, int64_t ld_dx, int accumulate, __nv_bfloat16* __restrict__ dx_bf16,
                               int64_t ld_b, int64_t lo_off, float* __restrict__ part) {
  constexpr int cols = NVEC * 128;
  __shared__ float red[3 * cols];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4 ag[NVEC], ab[NVEC], ac[NVEC];
#pragma unroll
  for (int i = 0; i < NVEC; ++i) ag[i] = ab[i] = ac[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 gm[NVEC];
#pragma unroll
  for (int i = 0; i < NVEC; ++i) gm[i] = __ldg(reinterpret_cast<const float4*>(gamma + (i * 32 + lane) * 4));
  const int64_t stride = (int64_t)gridDim.x * 8;
  for (int64_t row = (int64_t)blockIdx.x * 8 + warp; row < rows; row += stride) {
    const float* xr = x + row * ldx;
    const float* dyr = dy + row * ld_dy;
    float* dxr = dx + row * ld_dx;
    float4 v[NVEC], d[NVEC], pv[NVEC];
#pragma unroll
    for (int i = 0; i < NVEC; ++i) v[i] = *reinterpret_cast<const float4*>(xr + (i * 32 + lane) * 4);
#pragma unroll
    for (int i = 0; i < NVEC; ++i) d[i] = *reinterpret_cast<const float4*>(dyr + (i * 32 + lane) * 4);
    if (accumulate) {
#pragma unroll
      for (int i = 0; i < NVEC; ++i) pv[i] = *reinterpret_cast<const float4*>(dxr + (i * 32 + lane) * 4);
    }
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < NVEC; ++i) sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    const float mean = warp_sum(sum) * (1.0f / cols);
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < NVEC; ++i) {
      v[i].x -= mean, v[i].y -= mean, v[i].z -= mean, v[i].w -= mean;
      sq += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
    }
    const float rstd = rsqrtf(warp_sum(sq) * (1.0f / cols) + eps);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NVEC; ++i) {
      v[i].x *= rstd, v[i].y *= rstd, v[i].z *= rstd, v[i].w *= rstd;  // xhat
      ag[i].x += d[i].x * v[i].x, ag[i].y += d[i].y * v[i].y, ag[i].z += d[i].z * v[i].z, ag[i].w += d[i].w * v[i].w;
      ab[i].x += d[i].x, ab[i].y += d[i].y, ab[i].z += d[i].z, ab[i].w += d[i].w;
      d[i].x *= gm[i].x, d[i].y *= gm[i].y, d[i].z *= gm[i].z, d[i].w *= gm[i].w;  // g
      s1 += (d[i].x + d[i].y) + (d[i].z + d[i].w);
      s2 += (d[i].x * v[i].x + d[i].y * v[i].y) + (d[i].z * v[i].z + d[i].w * v[i].w);
    }
    s1 = warp_sum(s1) * (1.0f / cols);
    s2 = warp_sum(s2) * (1.0f / cols);
#pragma unroll
    for (int i = 0; i < NVEC; ++i) {
      const int c = (i * 32 + lane) * 4;
      float4 o;
      o.x = rstd * (d[i].x - s1 - v[i].x * s2);
      o.y = rstd * (d[i].y - s1 - v[i].y * s2);
      o.z = rstd * (d[i].z - s1 - v[i].z * s2);
      o.w = rstd * (d[i].w - s1 - v[i].w * s2);
      if (accumulate) o.x += pv[i].x, o.y += pv[i].y, o.z += pv[i].z, o.w += pv[i].w;
      *reinterpret_cast<float4*>(dxr + c) = o;
      ac[i].x += o.x, ac[i].y += o.y, ac[i].z += o.z, ac[i].w += o.w;
      if (dx_bf16) {
        __nv_bfloat16* b = dx_bf16 + row * ld_b + c;
        const uint32_t h0 = pack_bf16x2(o.x, o.y), h1 = pack_bf16x2(o.z, o.w);
        *reinterpret_cast<uint2*>(b) = make_uint2(h0, h1);
        if (lo_off > 0) {
          const float2 f0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&h0));
          const float2 f1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&h1));
          *reinterpret_cast<uint2*>(b + lo_off) =
              make_uint2(pack_bf16x2(o.x - f0.x, o.y - f0.y), pack_bf16x2(o.z - f1.x, o.w - f1.y));
        }
      }
    }
  }
  // block reduction in a fixed order: warp 0 stores, warps 1..7 add one after the other
  for (int w = 0; w < 8; ++w) {
    if (warp == w) {
#pragma unroll
      for (int i = 0; i < NVEC; ++i) {
        float4* r0 = reinterpret_cast<float4*>(red + (i * 32 + lane) * 4);
        float4* r1 = reinterpret_cast<float4*>(red + cols + (i * 32 + lane) * 4);
        float4* r2 = reinterpret_cast<float4*>(red + 2 * cols + (i * 32 + lane) * 4);
        if (w == 0) {
          *r0 = ag[i], *r1 = ab[i], *r2 = ac[i];
        } else {
          float4 t = *r0;
          t.x += ag[i].x, t.y += ag[i].y, t.z += ag[i].z, t.w += ag[i].w;
          *r0 = t;
          t = *r1;
          t.x += ab[i].x, t.y += ab[i].y, t.z += ab[i].z, t.w += ab[i].w;
          *r1 = t;
          t = *r2;
          t.x += ac[i].x, t.y += ac[i].y, t.z += ac[i].z, t.w += ac[i].w;
          *r2 = t;
        }
      }
    }
    __syncthreads();
  }
  for (int c = threadIdx.x; c < 3 * cols; c += 256) part[(size_t)blockIdx.x * 3 * cols + c] = red[c];
}

// out_dgb[0:2cols] (+)= sum_b part[b][0:2cols]; out_cs[0:cols] = sum_b part[b][2cols:3cols]
__global__ void ln_fused_final_kernel(const float* __restrict__ part, int nblocks, int cols,
                                      float* __restrict__ out_dgb, int accumulate,
                                      float* __restrict__ out_cs) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= 3 * cols) return;
  float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
  int k = 0;
  for (; k + 4 <= nblocks; k += 4) {
    t0 += part[(size_t)k * 3 * cols + c];
    t1 += part[(size_t)(k + 1) * 3 * cols + c];
    t2 += part[(size_t)(k + 2) * 3 * cols + c];
    t3 += part[(size_t)(k + 3) * 3 * cols + c];
  }
  for (; k < nblocks; ++k) t0 += part[(size_t)k * 3 * cols + c];
  const float t = (t0 + t1) + (t2 + t3);
  if (c < 2 * cols) out_dgb[c] = accumulate ? out_dgb[c] + t : t;
  else if (out_cs) out_cs[c - 2 * cols] = t;
}

// ------------------------------------------------------------------------------------------
// Full attention backward (CUDA cores, fp32 math), one CTA per (sequence, head), head_dim 64.
//   P = softmax(Q K^T / 8 [+causal]); dP = dO V^T; D_i = sum_j P_ij dP_ij; dS = P (dP - D) / 8
//   dQ = dS K; dK = dS^T Q; dV = P^T dO
// Q, K, V, dO live in shared memory as bf16 pairs with a 33-word row pitch (conflict-free for
// lane-per-row access); pass 1 sweeps query rows (dQ + row statistics), pass 2 sweeps key rows
// (dK, dV) re-deriving P from the saved statistics.
constexpr int kAbHd = 64;
// row pitch in 32-bit words: 64 bf16 + pad, or (fp32 parity mode) 64 floats + pad
template <bool F32> struct AbSt { static constexpr int pitch = F32 ? 65 : 33; };
template <bool F32>
__device__ __forceinline__ float2 ldpair(const uint32_t* row, int w) {
  if constexpr (F32) return make_float2(__uint_as_float(row[2 * w]), __uint_as_float(row[2 * w + 1]));
  else return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(row + w));
}
template <bool F32>
__device__ __forceinline__ void stpair(uint32_t* row, int w, float a, float b) {
  if constexpr (F32) row[2 * w] = __float_as_uint(a), row[2 * w + 1] = __float_as_uint(b);
  else row[w] = pack_bf16x2(a, b);
}
constexpr int kAbWarps = 8;
constexpr int kAbMaxT = 288;
constexpr int kAbChunks = kAbMaxT / 32;
constexpr int kAbMaxSmem = 227 * 1024;  // dynamic shared memory of one CTA

template <bool F32>
__device__ __forceinline__ float dot64(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b) {
  float acc = 0.f;
#pragma unroll
  for (int w = 0; w < 32; ++w) {
    const float2 x = ldpair<F32>(a, w), y = ldpair<F32>(b, w);
    acc += x.x * y.x + x.y * y.y;
  }
  return acc;
}

template <typename TI, typename TG, typename TO>
__global__ void __launch_bounds__(kAbWarps * 32, 1)
    attention_bwd_kernel(const TI* __restrict__ qkv, int64_t ld_qkv, int Tn, int H, int causal,
                         const TG* __restrict__ d_out, int64_t ld_do, TO* __restrict__ d_qkv,
                         int64_t ld_dqkv) {
  constexpr bool F32 = sizeof(TI) == 4;
  constexpr int kAbPitch = AbSt<F32>::pitch;
  extern __shared__ uint32_t smem_w[];
  uint32_t* sQ = smem_w;
  uint32_t* sK = sQ + Tn * kAbPitch;
  uint32_t* sV = sK + Tn * kAbPitch;
  uint32_t* sO = sV + Tn * kAbPitch;  // dO
  float* sM = reinterpret_cast<float*>(sO + Tn * kAbPitch);  // row max
  float* sL = sM + Tn;                                      // row sum
  float* sD = sL + Tn;                                      // D_i
  float* sBuf = sD + Tn;                                    // [warps][2][kAbMaxT]
  const int b = blockIdx.x / H, h = blockIdx.x % H, d = H * kAbHd;
  const TI* base = qkv + (int64_t)b * Tn * ld_qkv + h * kAbHd;
  const TG* dob = d_out + (int64_t)b * Tn * ld_do + h * kAbHd;
  TO* gb = d_qkv + (int64_t)b * Tn * ld_dqkv + h * kAbHd;
  for (int i = threadIdx.x; i < Tn * 32; i += blockDim.x) {
    const int r = i >> 5, w = i & 31;
    const TI* row = base + (int64_t)r * ld_qkv + 2 * w;
    stpair<F32>(sQ + r * kAbPitch, w, to_f(row[0]), to_f(row[1]));
    stpair<F32>(sK + r * kAbPitch, w, to_f(row[d]), to_f(row[d + 1]));
    stpair<F32>(sV + r * kAbPitch, w, to_f(row[2 * d]), to_f(row[2 * d + 1]));
    const TG* g = dob + (int64_t)r * ld_do + 2 * w;
    stpair<F32>(sO + r * kAbPitch, w, to_f(g[0]), to_f(g[1]));
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* bufA = sBuf + warp * 2 * kAbMaxT;
  float* bufB = bufA + kAbMaxT;
  const int nch = (Tn + 31) >> 5;
  // ---- pass 1: query rows -> statistics and dQ
  for (int i = warp; i < Tn; i += kAbWarps) {
    const int last = causal ? i : Tn - 1;
    float s[kAbChunks], dp[kAbChunks];
    float mx = -INFINITY;
#pragma unroll
    for (int c = 0; c < kAbChunks; ++c) {
      const int j = lane + 32 * c;
      s[c] = -INFINITY, dp[c] = 0.f;
      if (c < nch && j <= last) {
        s[c] = 0.125f * dot64<F32>(sQ + i * kAbPitch, sK + j * kAbPitch);
        dp[c] = dot64<F32>(sO + i * kAbPitch, sV + j * kAbPitch);
        mx = fmaxf(mx, s[c]);
      }
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int c = 0; c < kAbChunks; ++c) {
      s[c] = (s[c] == -INFINITY) ? 0.f : expf(s[c] - mx);
      sum += s[c];
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    float dsum = 0.f;
#pragma unroll
    for (int c = 0; c < kAbChunks; ++c) {
      s[c] *= inv;
      dsum += s[c] * dp[c];
    }
    dsum = warp_sum(dsum);
    if (lane == 0) sM[i] = mx, sL[i] = sum, sD[i] = dsum;
#pragma unroll
    for (int c = 0; c < kAbChunks; ++c) {
      const int j = lane + 32 * c;
      if (c < nch && j < kAbMaxT) bufA[j] = 0.125f * s[c] * (dp[c] - dsum);  // dS_ij
    }
    __syncwarp();
    float a0 = 0.f, a1 = 0.f;  // dQ_i[2*lane], dQ_i[2*lane+1]
    for (int j = 0; j <= last; ++j) {
      const float ds = bufA[j];
      const float2 kf = ldpair<F32>(sK + j * kAbPitch, lane);
      a0 += ds * kf.x;
      a1 += ds * kf.y;
    }
    TO* o = gb + (int64_t)i * ld_dqkv + 2 * lane;
    o[0] = from_f<TO>(a0);
    o[1] = from_f<TO>(a1);
    __syncwarp();
  }
  __syncthreads();
  // ---- pass 2: key rows -> dK, dV
  for (int j = warp; j < Tn; j += kAbWarps) {
    const int first = causal ? j : 0;
#pragma unroll
    for (int c = 0; c < kAbChunks; ++c) {
      const int i = lane + 32 * c;
      if (c < nch && i < kAbMaxT) {
        float p = 0.f, ds = 0.f;
        if (i < Tn && i >= first) {
          const float sc = 0.125f * dot64<F32>(sQ + i * kAbPitch, sK + j * kAbPitch);
          p = expf(sc - sM[i]) / sL[i];
          const float dpv = dot64<F32>(sO + i * kAbPitch, sV + j * kAbPitch);
          ds = 0.125f * p * (dpv - sD[i]);
        }
        bufA[i] = ds;
        bufB[i] = p;
      }
    }
    __syncwarp();
    float k0 = 0.f, k1 = 0.f, v0 = 0.f, v1 = 0.f;
    for (int i = first; i < Tn; ++i) {
      const float ds = bufA[i], p = bufB[i];
      const float2 qf = ldpair<F32>(sQ + i * kAbPitch, lane);
      const float2 of = ldpair<F32>(sO + i * kAbPitch, lane);
      k0 += ds * qf.x, k1 += ds * qf.y;
      v0 += p * of.x, v1 += p * of.y;
    }
    TO* o = gb + (int64_t)j * ld_dqkv + 2 * lane;
    o[d] = from_f<TO>(k0);
    o[d + 1] = from_f<TO>(k1);
    o[2 * d] = from_f<TO>(v0);
    o[2 * d + 1] = from_f<TO>(v1);
    __syncwarp();
  }
}

template <typename TI, typename TG, typename TO>
static int launch_attention_bwd(const void* qkv, int64_t ld_qkv, int B, int T, int H, int causal,
                                const void* d_out, int64_t ld_do, void* d_qkv, int64_t ld_dqkv,
                                cudaStream_t s) {
  const size_t smem = sizeof(uint32_t) * 4 * (size_t)T * AbSt<sizeof(TI) == 4>::pitch + sizeof(float) * 3 * (size_t)T +
                      sizeof(float) * kAbWarps * 2 * kAbMaxT;
  HBA_REQUIRE(smem <= kAbMaxSmem, "hba_attention_bwd: T=%d needs %zu bytes of shared memory (max %d; fp32 qkv: T <= 203)",
              T, smem, kAbMaxSmem);
  static SmemAttr attr;
  HBA_CHECK(ensure_dyn_smem(attention_bwd_kernel<TI, TG, TO>, smem, attr, "attention_bwd_kernel"));
  attention_bwd_kernel<TI, TG, TO><<<B * H, kAbWarps * 32, smem, s>>>(
      static_cast<const TI*>(qkv), ld_qkv, T, H, causal, static_cast<const TG*>(d_out), ld_do,
      static_cast<TO*>(d_qkv), ld_dqkv);
  return check_launch("attention_bwd_kernel");
}

}  // namespace hba

using namespace hba;

extern "C" int hba_colsum(const void* x, int32_t dtype, int64_t rows, int32_t cols, int64_t ld,
                          float* out, int32_t accumulate, float* workspace, void* stream) {
  HBA_REQUIRE(x && out && workspace && rows > 0 && cols > 0, "hba_colsum: bad arguments");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  dim3 grid((cols + 31) / 32, kCsChunks), block(32, 8);
  if (dtype == HBA_DT_F32)
    colsum_partial_kernel<float><<<grid, block, 0, s>>>(static_cast<const float*>(x), rows, cols, ld, workspace);
  else if (dtype == HBA_DT_BF16)
    colsum_partial_kernel<__nv_bfloat16><<<grid, block, 0, s>>>(static_cast<const __nv_bfloat16*>(x), rows, cols, ld, workspace);
  else {
    set_error("hba_colsum: unknown dtype %d", dtype);
    return HBA_ERR_ARG;
  }
  HBA_CHECK(check_launch("colsum_partial_kernel"));
  colsum_final_kernel<<<(cols + 255) / 256, 256, 0, s>>>(workspace, cols, out, accumulate);
  return check_launch("colsum_final_kernel");
}

extern "C" int hba_layernorm_param_grad(const float* dy, int64_t ld_dy, const float* x, int64_t rows,
                                        int32_t cols, int64_t ldx, int64_t row_step, float eps,
                                        float* dgamma_dbeta, int32_t accumulate, float* workspace,
                                        void* stream) {
  HBA_REQUIRE(dy && x && dgamma_dbeta && workspace && rows > 0 && cols > 0 && cols % 4 == 0,
              "hba_layernorm_param_grad: bad arguments");
  HBA_REQUIRE(ldx % 4 == 0 && aligned16(x),
              "hba_layernorm_param_grad: x rows are read as float4: x must be 16-byte aligned and ldx a multiple of 4");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* stats = workspace;                 // [rows, 2]
  float* partial = workspace + 2 * rows;    // [chunks, 2*cols]
  ln_stats_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(x, rows, cols, ldx, row_step < 1 ? 1 : row_step, eps, stats);
  HBA_CHECK(check_launch("ln_stats_kernel"));
  dim3 grid((cols + 31) / 32, kCsChunks), block(32, 8);
  ln_param_partial_kernel<<<grid, block, 0, s>>>(dy, ld_dy, x, ldx, row_step < 1 ? 1 : row_step, stats, rows, cols, partial);
  HBA_CHECK(check_launch("ln_param_partial_kernel"));
  colsum_final_kernel<<<(2 * cols + 255) / 256, 256, 0, s>>>(partial, 2 * cols, dgamma_dbeta, accumulate);
  return check_launch("colsum_final_kernel");
}

extern "C" int hba_attention_bwd(const void* qkv, int32_t qkv_dtype, int64_t ld_qkv, int32_t B,
                                 int32_t T, int32_t H, int32_t causal, const void* d_out,
                                 int32_t do_dtype, int64_t ld_do, void* d_qkv, int32_t dq_dtype,
                                 int64_t ld_dqkv, void* stream) {
  HBA_REQUIRE(qkv && d_out && d_qkv && B > 0 && T > 0 && H > 0, "hba_attention_bwd: bad arguments");
  HBA_REQUIRE(T <= kAbMaxT, "hba_attention_bwd: T=%d exceeds %d", T, kAbMaxT);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (qkv_dtype == HBA_DT_BF16 && do_dtype == HBA_DT_BF16 && dq_dtype == HBA_DT_BF16)
    return launch_attention_bwd<__nv_bfloat16, __nv_bfloat16, __nv_bfloat16>(qkv, ld_qkv, B, T, H, causal, d_out, ld_do, d_qkv, ld_dqkv, s);
  if (qkv_dtype == HBA_DT_BF16 && do_dtype == HBA_DT_F32 && dq_dtype == HBA_DT_BF16)
    return launch_attention_bwd<__nv_bfloat16, float, __nv_bfloat16>(qkv, ld_qkv, B, T, H, causal, d_out, ld_do, d_qkv, ld_dqkv, s);
  if (qkv_dtype == HBA_DT_F32 && do_dtype == HBA_DT_F32 && dq_dtype == HBA_DT_F32)
    return launch_attention_bwd<float, float, float>(qkv, ld_qkv, B, T, H, causal, d_out, ld_do, d_qkv, ld_dqkv, s);
  set_error("hba_attention_bwd: unsupported dtype combination (%d, %d, %d)", qkv_dtype, do_dtype, dq_dtype);
  return HBA_ERR_ARG;
}

extern "C" int hba_layernorm_bwd_fused(const float* dy, int64_t ld_dy, const float* x, int64_t rows,
                                       int32_t cols, int64_t ldx, const float* gamma, float eps,
                                       float* dx, int64_t ld_dx, int32_t accumulate, void* dx_bf16,
                                       int64_t ld_b, int64_t lo_off, float* dgamma_dbeta,
                                       int32_t accumulate_params, float* dx_colsum, float* workspace,
                                       void* stream) {
  HBA_REQUIRE(dy && x && gamma && dx && dgamma_dbeta && workspace && rows > 0, "hba_layernorm_bwd_fused: bad arguments");
  HBA_REQUIRE(ldx % 4 == 0 && ld_dy % 4 == 0 && ld_dx % 4 == 0 && ld_b % 4 == 0 && lo_off % 4 == 0,
              "hba_layernorm_bwd_fused: leading dimensions must be multiples of 4");
  HBA_REQUIRE(aligned16(dy) && aligned16(x) && aligned16(gamma) && aligned16(dx) && ((uintptr_t)dx_bf16 & 7) == 0,
              "hba_layernorm_bwd_fused: dy, x, gamma and dx must be 16-byte aligned (float4), dx_bf16 8-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int blocks = 2 * num_sms();
  if ((int64_t)blocks * 8 > rows) blocks = (int)((rows + 7) / 8);
  __nv_bfloat16* b = static_cast<__nv_bfloat16*>(dx_bf16);
#define HBA_LN_FUSED(NV)                                                                            \
  layernorm_bwd_fused_kernel<NV><<<blocks, 256, 0, s>>>(dy, ld_dy, x, rows, ldx, gamma, eps, dx, ld_dx, \
                                                        accumulate, b, ld_b, lo_off, workspace)
  switch (cols) {
    case 128: HBA_LN_FUSED(1); break;
    case 256: HBA_LN_FUSED(2); break;
    case 512: HBA_LN_FUSED(4); break;
    case 768: HBA_LN_FUSED(6); break;
    case 1024: HBA_LN_FUSED(8); break;
    default:
      set_error("hba_layernorm_bwd_fused: cols=%d (supported: 128, 256, 512, 768, 1024)", cols);
      return HBA_ERR_ARG;
  }
#undef HBA_LN_FUSED
  HBA_CHECK(check_launch("layernorm_bwd_fused_kernel"));
  ln_fused_final_kernel<<<(3 * cols + 255) / 256, 256, 0, s>>>(workspace, blocks, cols, dgamma_dbeta,
                                                             accumulate_params, dx_colsum);
  return check_launch("ln_fused_final_kernel");
}
