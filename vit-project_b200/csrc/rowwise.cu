// Bandwidth-bound row-wise kernels of the CLIP-HBA towers: operand staging (fp32 -> bf16 hi/lo),
// LayerNorm forward/backward, patch im2col, token assembly + ln_pre, text embedding, row gathers.
// All are one-warp-per-row or grid-stride kernels with 128-bit accesses; bound: HBM.
#include "common.cuh"

namespace hba {

// ---------------------------------------------------------------------------------------------
// fp32 -> bf16 hi (+ lo) staging, optionally transposed (32x32 smem tile transpose)
__global__ void split_bf16_kernel(const float* __restrict__ in, int64_t rows, int64_t cols,
                                  int64_t ld_in, __nv_bfloat16* __restrict__ out, int64_t ld_out,
                                  int64_t lo_off) {
  const int64_t n4 = cols / 4;
  const int64_t total = rows * n4;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / n4, c = (i % n4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(in + r * ld_in + c);
    __nv_bfloat16 h0, h1, h2, h3, l0, l1, l2, l3;
    split_bf16(v.x, h0, l0), split_bf16(v.y, h1, l1), split_bf16(v.z, h2, l2),
        split_bf16(v.w, h3, l3);
    __nv_bfloat16* o = out + r * ld_out + c;
    *reinterpret_cast<__nv_bfloat162*>(o) = __nv_bfloat162(h0, h1);
    *reinterpret_cast<__nv_bfloat162*>(o + 2) = __nv_bfloat162(h2, h3);
    if (lo_off > 0) {
      *reinterpret_cast<__nv_bfloat162*>(o + lo_off) = __nv_bfloat162(l0, l1);
      *reinterpret_cast<__nv_bfloat162*>(o + lo_off + 2) = __nv_bfloat162(l2, l3);
    }
  }
}

__global__ void split_bf16_transpose_kernel(const float* __restrict__ in, int64_t rows,
                                            int64_t cols, int64_t ld_in,
                                            __nv_bfloat16* __restrict__ out, int64_t ld_out,
                                            int64_t lo_off) {
  __shared__ float tile[32][33];
  const int64_t r0 = (int64_t)blockIdx.y * 32, c0 = (int64_t)blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? in[r * ld_in + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t c = c0 + i, r = r0 + threadIdx.x;  // out[c, r]
    if (c < cols && r < rows) {
      __nv_bfloat16 h, l;
      split_bf16(tile[threadIdx.x][i], h, l);
      out[c * ld_out + r] = h;
      if (lo_off > 0) out[c * ld_out + lo_off + r] = l;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// LayerNorm: one warp per row; the row lives in registers (cols <= 32 * 4 * kMaxVec)
constexpr int kLnMaxVec = 8;  // up to 1024 columns

__device__ __forceinline__ void ln_store(float4 y, int c, float* y_f32, __nv_bfloat16* y_bf16,
                                         int64_t lo_off) {
  if (y_f32) *reinterpret_cast<float4*>(y_f32 + c) = y;
  if (y_bf16) {
    __nv_bfloat16 h0, h1, h2, h3, l0, l1, l2, l3;
    split_bf16(y.x, h0, l0), split_bf16(y.y, h1, l1), split_bf16(y.z, h2, l2),
        split_bf16(y.w, h3, l3);
    // one 8-byte store per lane: a warp writes 256 contiguous bytes per instruction
    __nv_bfloat162 p0(h0, h1), p1(h2, h3);
    *reinterpret_cast<uint2*>(y_bf16 + c) =
        make_uint2(*reinterpret_cast<uint32_t*>(&p0), *reinterpret_cast<uint32_t*>(&p1));
    if (lo_off > 0) {
      __nv_bfloat162 q0(l0, l1), q1(l2, l3);
      *reinterpret_cast<uint2*>(y_bf16 + lo_off + c) =
          make_uint2(*reinterpret_cast<uint32_t*>(&q0), *reinterpret_cast<uint32_t*>(&q1));
    }
  }
}

__global__ void __launch_bounds__(256)
    layernorm_fwd_kernel(const float* __restrict__ x, int64_t rows, int cols, int64_t ldx,
                         int64_t row_step, const float* __restrict__ gamma,
                         const float* __restrict__ beta, float eps, float* __restrict__ y_f32,
                         int64_t ld_yf, __nv_bfloat16* __restrict__ y_bf16, int64_t ld_yb,
                         int64_t lo_off) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + row * row_step * ldx;
  const int nvec = cols / 128;  // float4 per lane
  float4 v[kLnMaxVec];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i)
    if (i < nvec) {
      v[i] = *reinterpret_cast<const float4*>(xr + (i * 32 + lane) * 4);
      sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  const float mean = warp_sum(sum) / cols;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i)
    if (i < nvec) {
      const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
      sq += (a * a + b * b) + (c * c + d * d);
    }
  const float rstd = rsqrtf(warp_sum(sq) / cols + eps);
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i)
    if (i < nvec) {
      const int c = (i * 32 + lane) * 4;
      const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma + c));
      const float4 bt = __ldg(reinterpret_cast<const float4*>(beta + c));
      float4 y;
      y.x = (v[i].x - mean) * rstd * gm.x + bt.x;
      y.y = (v[i].y - mean) * rstd * gm.y + bt.y;
      y.z = (v[i].z - mean) * rstd * gm.z + bt.z;
      y.w = (v[i].w - mean) * rstd * gm.w + bt.w;
      ln_store(y, c, y_f32 ? y_f32 + row * ld_yf : nullptr, y_bf16 ? y_bf16 + row * ld_yb : nullptr,
               lo_off);
    }
}

// ---------------------------------------------------------------------------------------------
// LayerNorm forward, streaming form for the big activations (>= 1024 rows; the 74 launches of a CLIP-HBA step
// are 8224 x 1024 / 5082 x 768): one persistent CTA per SM owns a contiguous range of rows and pulls them
// through a ring of shared-memory stages with bulk asynchronous copies (cp.async.bulk, one per row, completion
// on an mbarrier), so that ~190 KB of loads are in flight per SM independently of register pressure and the
// grid has no second wave.  Warp w of the 8 consumer warps normalises row w of a stage out of shared memory;
// the arithmetic (per-lane partial sums in the same order, xor-shuffle reductions, two-pass variance) is the
// one of layernorm_fwd_kernel, so both kernels produce identical bits.
// 24 consumer warps: with 8 the kernel was issue-latency bound (ncu: 2 warps per scheduler, 0.19 IPC per warp,
// 39 % issue-active, DRAM at 26 % of peak, 16.2 us cold); a row costs ~830 warp instructions, i.e. 46 k per SM.
constexpr int kLnsRows = 24;        // rows per stage = consumer warps
constexpr int kLnsThreads = 32 * (kLnsRows + 1);
constexpr int kLnsMaxStages = 8;

__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

__global__ void __launch_bounds__(kLnsThreads, 1)
    layernorm_fwd_stream_kernel(const float* __restrict__ x, int64_t rows, int cols, int64_t ldx,
                                int64_t row_step, const float* __restrict__ gamma,
                                const float* __restrict__ beta, float eps, float* __restrict__ y_f32,
                                int64_t ld_yf, __nv_bfloat16* __restrict__ y_bf16, int64_t ld_yb,
                                int64_t lo_off, int stages) {
  extern __shared__ __align__(128) uint8_t lns_smem[];
  float* s_gamma = reinterpret_cast<float*>(lns_smem);
  float* s_beta = s_gamma + cols;
  float* s_rows = s_beta + cols;                                    // [stages][kLnsRows][cols]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_rows + (size_t)stages * kLnsRows * cols);
  uint64_t* empty_bar = full_bar + kLnsMaxStages;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row_begin = rows * blockIdx.x / gridDim.x, row_end = rows * (blockIdx.x + 1) / gridDim.x;
  const int n_iters = (int)((row_end - row_begin + kLnsRows - 1) / kLnsRows);
  if (threadIdx.x == 0) {
    for (int i = 0; i < stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], kLnsRows);
    }
    mbar_fence_init();
  }
  for (int c = threadIdx.x * 4; c < cols; c += kLnsThreads * 4) {
    *reinterpret_cast<float4*>(s_gamma + c) = __ldg(reinterpret_cast<const float4*>(gamma + c));
    *reinterpret_cast<float4*>(s_beta + c) = __ldg(reinterpret_cast<const float4*>(beta + c));
  }
  __syncthreads();
  const uint32_t row_bytes = (uint32_t)cols * 4u;
  if (warp == kLnsRows) {
    if (lane == 0) {
      for (int it = 0; it < n_iters; ++it) {
        const int st = it % stages;
        if (it >= stages) mbar_wait(&empty_bar[st], ((it / stages) - 1) & 1);
        const int64_t r0 = row_begin + (int64_t)it * kLnsRows;
        const int n = (int)min((int64_t)kLnsRows, row_end - r0);
        mbar_arrive_expect_tx(&full_bar[st], n * row_bytes);
        for (int r = 0; r < n; ++r)
          bulk_load_1d(s_rows + ((size_t)st * kLnsRows + r) * cols, x + (r0 + r) * row_step * ldx, row_bytes,
                       &full_bar[st]);
      }
    }
    return;
  }
  const int nvec = cols / 128;  // float4 per lane
  for (int it = 0; it < n_iters; ++it) {
    const int st = it % stages;
    mbar_wait(&full_bar[st], (it / stages) & 1);
    const int64_t row = row_begin + (int64_t)it * kLnsRows + warp;
    if (row < row_end) {
      const float* xr = s_rows + ((size_t)st * kLnsRows + warp) * cols;
      float4 v[kLnMaxVec];
      float sum = 0.f;
#pragma unroll
      for (int i = 0; i < kLnMaxVec; ++i)
        if (i < nvec) {
          v[i] = *reinterpret_cast<const float4*>(xr + (i * 32 + lane) * 4);
          sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
        }
      const float mean = warp_sum(sum) / cols;
      float sq = 0.f;
#pragma unroll
      for (int i = 0; i < kLnMaxVec; ++i)
        if (i < nvec) {
          const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
          sq += (a * a + b * b) + (c * c + d * d);
        }
      const float rstd = rsqrtf(warp_sum(sq) / cols + eps);
#pragma unroll
      for (int i = 0; i < kLnMaxVec; ++i)
        if (i < nvec) {
          const int c = (i * 32 + lane) * 4;
          const float4 gm = *reinterpret_cast<const float4*>(s_gamma + c);
          const float4 bt = *reinterpret_cast<const float4*>(s_beta + c);
          float4 y;
          y.x = (v[i].x - mean) * rstd * gm.x + bt.x;
          y.y = (v[i].y - mean) * rstd * gm.y + bt.y;
          y.z = (v[i].z - mean) * rstd * gm.z + bt.z;
          y.w = (v[i].w - mean) * rstd * gm.w + bt.w;
          ln_store(y, c, y_f32 ? y_f32 + row * ld_yf : nullptr, y_bf16 ? y_bf16 + row * ld_yb : nullptr,
                   lo_off);
        }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[st]);   // this warp's row of the stage has been read
  }
}

// dx = rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma
__global__ void __launch_bounds__(256)
    layernorm_bwd_kernel(const float* __restrict__ dy, int64_t ld_dy, const float* __restrict__ x,
                         int64_t rows, int cols, int64_t ldx, int64_t row_step,
                         const float* __restrict__ gamma, float eps, float* __restrict__ dx,
                         int64_t ld_dx, int accumulate) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + row * row_step * ldx;
  const float* dyr = dy + row * ld_dy;
  float* dxr = dx + row * ld_dx;
  const int nvec = cols / 128;
  float4 v[kLnMaxVec], gg[kLnMaxVec];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i)
    if (i < nvec) {
      v[i] = *reinterpret_cast<const float4*>(xr + (i * 32 + lane) * 4);
      sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  const float mean = warp_sum(sum) / cols;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i)
    if (i < nvec) {
      v[i].x -= mean, v[i].y -= mean, v[i].z -= mean, v[i].w -= mean;
      sq += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
    }
  const float rstd = rsqrtf(warp_sum(sq) / cols + eps);
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i)
    if (i < nvec) {
      const int c = (i * 32 + lane) * 4;
      const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma + c));
      const float4 d = *reinterpret_cast<const float4*>(dyr + c);
      v[i].x *= rstd, v[i].y *= rstd, v[i].z *= rstd, v[i].w *= rstd;  // xhat
      gg[i] = make_float4(d.x * gm.x, d.y * gm.y, d.z * gm.z, d.w * gm.w);
      s1 += (gg[i].x + gg[i].y) + (gg[i].z + gg[i].w);
      s2 += (gg[i].x * v[i].x + gg[i].y * v[i].y) + (gg[i].z * v[i].z + gg[i].w * v[i].w);
    }
  s1 = warp_sum(s1) / cols;
  s2 = warp_sum(s2) / cols;
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i)
    if (i < nvec) {
      const int c = (i * 32 + lane) * 4;
      float4 o;
      o.x = rstd * (gg[i].x - s1 - v[i].x * s2);
      o.y = rstd * (gg[i].y - s1 - v[i].y * s2);
      o.z = rstd * (gg[i].z - s1 - v[i].z * s2);
      o.w = rstd * (gg[i].w - s1 - v[i].w * s2);
      if (accumulate) {
        const float4 p = *reinterpret_cast<const float4*>(dxr + c);
        o.x += p.x, o.y += p.y, o.z += p.z, o.w += p.w;
      }
      *reinterpret_cast<float4*>(dxr + c) = o;
    }
}

// ---------------------------------------------------------------------------------------------
// im2col for a PxP / stride-P convolution: one warp per patch row
__global__ void im2col_kernel(const float* __restrict__ image, int B, int H, int W, int P,
                              __nv_bfloat16* __restrict__ out, int64_t ld_out, int64_t lo_off) {
  const int gw = W / P, gh = H / P;
  const int64_t patch = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (patch >= (int64_t)B * gh * gw) return;
  const int lane = threadIdx.x & 31;
  const int b = patch / (gh * gw), pr = (patch / gw) % gh, pc = patch % gw;
  const int kk = 3 * P * P;
  __nv_bfloat16* o = out + patch * ld_out;
  // hi part: columns [0, hi_end); lo part: columns lo_off + [0, lo_end) - both zero past 3*P*P, neither past ld_out
  const int64_t hi_end = lo_off > 0 ? lo_off : ld_out, lo_end = lo_off > 0 ? ld_out - lo_off : 0;
  for (int64_t k = lane; k < hi_end || k < lo_end; k += 32) {
    float v = 0.f;
    if (k < kk) {
      const int c = k / (P * P), py = (k / P) % P, px = k % P;
      v = image[(((int64_t)b * 3 + c) * H + pr * P + py) * W + pc * P + px];
    }
    __nv_bfloat16 h, l;
    split_bf16(v, h, l);
    if (k < hi_end) o[k] = h;
    if (k < lo_end) o[lo_off + k] = l;
  }
}

// x[b,t,:] = ln_pre( (t == 0 ? cls : conv[b, t-1, :]) + pos[t] ); one warp per token row
__global__ void __launch_bounds__(256)
    assemble_tokens_ln_kernel(const float* __restrict__ conv, int B, int n_patches, int width,
                              const float* __restrict__ cls, const float* __restrict__ pos,
                              const float* __restrict__ gamma, const float* __restrict__ beta,
                              float eps, float* __restrict__ x_out) {
  const int lane = threadIdx.x & 31;
  const int T = n_patches + 1;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= (int64_t)B * T) return;
  const int b = row / T, t = row % T;
  const float* src = (t == 0) ? cls : conv + ((int64_t)b * n_patches + (t - 1)) * width;
  const float* pr = pos + (int64_t)t * width;
  const int nvec = width / 128;
  float4 v[kLnMaxVec];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i)
    if (i < nvec) {
      const int c = (i * 32 + lane) * 4;
      const float4 a = *reinterpret_cast<const float4*>(src + c);
      const float4 p = __ldg(reinterpret_cast<const float4*>(pr + c));
      v[i] = make_float4(a.x + p.x, a.y + p.y, a.z + p.z, a.w + p.w);
      sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  const float mean = warp_sum(sum) / width;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i)
    if (i < nvec) {
      const float a = v[i].x - mean, b2 = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
      sq += (a * a + b2 * b2) + (c * c + d * d);
    }
  const float rstd = rsqrtf(warp_sum(sq) / width + eps);
  float* o = x_out + row * width;
  if (gamma == nullptr) {  // no ln_pre (timm ViT): plain token assembly
#pragma unroll
    for (int i = 0; i < kLnMaxVec; ++i)
      if (i < nvec) *reinterpret_cast<float4*>(o + (i * 32 + lane) * 4) = v[i];
    return;
  }
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i)
    if (i < nvec) {
      const int c = (i * 32 + lane) * 4;
      const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma + c));
      const float4 bt = __ldg(reinterpret_cast<const float4*>(beta + c));
      float4 y;
      y.x = (v[i].x - mean) * rstd * gm.x + bt.x;
      y.y = (v[i].y - mean) * rstd * gm.y + bt.y;
      y.z = (v[i].z - mean) * rstd * gm.z + bt.z;
      y.w = (v[i].w - mean) * rstd * gm.w + bt.w;
      *reinterpret_cast<float4*>(o + c) = y;
    }
}

__global__ void embed_tokens_kernel(const int64_t* __restrict__ tokens, int S, int T, int width,
                                    const float* __restrict__ table, const float* __restrict__ pos,
                                    float* __restrict__ x_out) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= (int64_t)S * T) return;
  const int lane = threadIdx.x & 31;
  const int t = row % T;
  const float* e = table + tokens[row] * (int64_t)width;
  const float* p = pos + (int64_t)t * width;
  float* o = x_out + row * width;
  for (int c = lane * 4; c < width; c += 128) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(e + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p + c));
    *reinterpret_cast<float4*>(o + c) = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  }
}

__global__ void gather_rows_kernel(const float* __restrict__ in, int64_t ld_in,
                                   const int64_t* __restrict__ idx, int n, int cols,
                                   float* __restrict__ out, int64_t ld_out) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const int lane = threadIdx.x & 31;
  const float* s = in + idx[row] * ld_in;
  float* o = out + row * ld_out;
  for (int c = lane; c < cols; c += 32) o[c] = s[c];
}

// dst[r * dst_row_step, :] += src[r, :]
__global__ void add_rows_kernel(float* __restrict__ dst, int64_t ld_dst, int64_t dst_row_step,
                                const float* __restrict__ src, int64_t ld_src, int64_t rows,
                                int cols) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  float* d = dst + row * dst_row_step * ld_dst;
  const float* s = src + row * ld_src;
  for (int c = lane; c < cols; c += 32) d[c] += s[c];
}

__global__ void nonfinite_flag_kernel(const float* __restrict__ x, int64_t n, int* flag) {
  bool bad = false;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    bad |= !isfinite(x[i]);
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}

static inline int grid_for(int64_t work, int per_block, int cap_mult = 16) {
  int64_t g = (work + per_block - 1) / per_block;
  const int64_t cap = (int64_t)num_sms() * cap_mult;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace hba

using namespace hba;

extern "C" int hba_split_bf16(const float* in, int64_t rows, int64_t cols, int64_t ld_in, void* out,
                              int64_t ld_out, int64_t lo_off, int transpose, void* stream) {
  HBA_REQUIRE(in && out && rows > 0 && cols > 0, "hba_split_bf16: bad arguments");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!transpose) {
    HBA_REQUIRE(cols % 4 == 0 && ld_in % 4 == 0 && ld_out % 2 == 0 && lo_off % 2 == 0 &&
                    ((uintptr_t)in & 15) == 0 && ((uintptr_t)out & 3) == 0,
                "hba_split_bf16: cols/ld must be multiples of 4 and pointers aligned");
    split_bf16_kernel<<<grid_for(rows * (cols / 4), 256), 256, 0, s>>>(
        in, rows, cols, ld_in, static_cast<__nv_bfloat16*>(out), ld_out, lo_off);
  } else {
    dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((rows + 31) / 32));
    split_bf16_transpose_kernel<<<grid, dim3(32, 8), 0, s>>>(
        in, rows, cols, ld_in, static_cast<__nv_bfloat16*>(out), ld_out, lo_off);
  }
  return check_launch("hba_split_bf16");
}

extern "C" int hba_layernorm_fwd(const float* x, int64_t rows, int32_t cols, int64_t ldx,
                                 int64_t row_step, const float* gamma, const float* beta, float eps,
                                 float* y_f32, int64_t ld_yf, void* y_bf16, int64_t ld_yb,
                                 int64_t lo_off, void* stream) {
  HBA_REQUIRE(x && gamma && beta && (y_f32 || y_bf16) && rows > 0, "hba_layernorm_fwd: bad arguments");
  HBA_REQUIRE(cols % 128 == 0 && cols <= 128 * kLnMaxVec, "hba_layernorm_fwd: cols=%d must be a multiple of 128 and <= %d", cols, 128 * kLnMaxVec);
  HBA_REQUIRE(ldx % 4 == 0 && ld_yf % 4 == 0 && ld_yb % 4 == 0 && lo_off % 4 == 0 && ((uintptr_t)y_bf16 & 7) == 0, "hba_layernorm_fwd: leading dimensions must keep 16-byte (fp32) / 8-byte (bf16) alignment");
  HBA_REQUIRE(aligned16(x) && aligned16(gamma) && aligned16(beta) && aligned16(y_f32),
              "hba_layernorm_fwd: x, gamma, beta and y_f32 are read / written as float4 and must be 16-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (row_step < 1) row_step = 1;
  if (rows >= 1024) {
    // streaming form: persistent CTAs, rows staged through shared memory by bulk asynchronous copies
    int stages = (int)((220 * 1024 - 2 * cols * 4 - 256) / ((size_t)kLnsRows * cols * 4));
    if (stages > kLnsMaxStages) stages = kLnsMaxStages;
    const size_t smem = (size_t)2 * cols * 4 + (size_t)stages * kLnsRows * cols * 4 + 2 * kLnsMaxStages * 8;
    static SmemAttr attr;
    HBA_CHECK(ensure_dyn_smem(layernorm_fwd_stream_kernel, smem, attr, "layernorm_fwd_stream_kernel"));
    int grid = num_sms();
    if ((int64_t)grid * kLnsRows > rows) grid = (int)((rows + kLnsRows - 1) / kLnsRows);
    layernorm_fwd_stream_kernel<<<grid, kLnsThreads, smem, s>>>(x, rows, cols, ldx, row_step, gamma, beta, eps, y_f32,
                                                                ld_yf, static_cast<__nv_bfloat16*>(y_bf16), ld_yb,
                                                                lo_off, stages);
    return check_launch("hba_layernorm_fwd (stream)");
  }
  layernorm_fwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(
      x, rows, cols, ldx, row_step, gamma, beta, eps, y_f32, ld_yf,
      static_cast<__nv_bfloat16*>(y_bf16), ld_yb, lo_off);
  return check_launch("hba_layernorm_fwd");
}

extern "C" int hba_layernorm_bwd(const float* dy, int64_t ld_dy, const float* x, int64_t rows,
                                 int32_t cols, int64_t ldx, int64_t row_step, const float* gamma,
                                 float eps, float* dx, int64_t ld_dx, int accumulate, void* stream) {
  HBA_REQUIRE(dy && x && gamma && dx && rows > 0, "hba_layernorm_bwd: bad arguments");
  HBA_REQUIRE(cols % 128 == 0 && cols <= 128 * kLnMaxVec, "hba_layernorm_bwd: cols=%d must be a multiple of 128 and <= %d", cols, 128 * kLnMaxVec);
  HBA_REQUIRE(ldx % 4 == 0 && ld_dy % 4 == 0 && ld_dx % 4 == 0, "hba_layernorm_bwd: leading dimensions must be multiples of 4");
  HBA_REQUIRE(aligned16(dy) && aligned16(x) && aligned16(gamma) && aligned16(dx),
              "hba_layernorm_bwd: dy, x, gamma and dx are accessed as float4 and must be 16-byte aligned");
  layernorm_bwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      dy, ld_dy, x, rows, cols, ldx, row_step < 1 ? 1 : row_step, gamma, eps, dx, ld_dx, accumulate);
  return check_launch("hba_layernorm_bwd");
}

extern "C" int hba_im2col_patches(const float* image, int32_t B, int32_t H, int32_t W, int32_t P,
                                  void* out, int64_t ld_out, int64_t lo_off, void* stream) {
  HBA_REQUIRE(image && out && B > 0 && P > 0 && H % P == 0 && W % P == 0, "hba_im2col_patches: bad arguments");
  HBA_REQUIRE((lo_off == 0 ? ld_out : lo_off) >= 3 * P * P && (lo_off == 0 || ld_out - lo_off >= 3 * P * P),
              "hba_im2col_patches: row too short for 3*P*P columns");
  const int64_t patches = (int64_t)B * (H / P) * (W / P);
  im2col_kernel<<<(unsigned)((patches + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      image, B, H, W, P, static_cast<__nv_bfloat16*>(out), ld_out, lo_off);
  return check_launch("hba_im2col_patches");
}

extern "C" int hba_assemble_tokens_ln(const float* conv, int32_t B, int32_t n_patches,
                                      int32_t width, const float* cls, const float* pos,
                                      const float* gamma, const float* beta, float eps,
                                      float* x_out, void* stream) {
  HBA_REQUIRE(conv && cls && pos && x_out && B > 0 && (!gamma == !beta), "hba_assemble_tokens_ln: bad arguments");
  HBA_REQUIRE(width % 128 == 0 && width <= 128 * kLnMaxVec, "hba_assemble_tokens_ln: width=%d unsupported", width);
  HBA_REQUIRE(aligned16(conv) && aligned16(cls) && aligned16(pos) && aligned16(gamma) && aligned16(beta) && aligned16(x_out),
              "hba_assemble_tokens_ln: conv, cls, pos, gamma, beta and x_out are accessed as float4 and must be 16-byte aligned");
  const int64_t rows = (int64_t)B * (n_patches + 1);
  assemble_tokens_ln_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      conv, B, n_patches, width, cls, pos, gamma, beta, eps, x_out);
  return check_launch("hba_assemble_tokens_ln");
}

extern "C" int hba_embed_tokens(const int64_t* tokens, int32_t S, int32_t T, int32_t width,
                                const float* table, const float* pos, float* x_out, void* stream) {
  HBA_REQUIRE(tokens && table && pos && x_out && S > 0 && T > 0 && width % 4 == 0, "hba_embed_tokens: bad arguments");
  HBA_REQUIRE(aligned16(table) && aligned16(pos) && aligned16(x_out),
              "hba_embed_tokens: table, pos and x_out are accessed as float4 and must be 16-byte aligned");
  const int64_t rows = (int64_t)S * T;
  embed_tokens_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      tokens, S, T, width, table, pos, x_out);
  return check_launch("hba_embed_tokens");
}

extern "C" int hba_gather_rows(const float* in, int64_t ld_in, const int64_t* idx, int32_t n,
                               int32_t cols, float* out, int64_t ld_out, void* stream) {
  HBA_REQUIRE(in && idx && out && n > 0 && cols > 0, "hba_gather_rows: bad arguments");
  gather_rows_kernel<<<(unsigned)((n + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      in, ld_in, idx, n, cols, out, ld_out);
  return check_launch("hba_gather_rows");
}

extern "C" int hba_add_rows(float* dst, int64_t ld_dst, int64_t dst_row_step, const float* src,
                            int64_t ld_src, int64_t rows, int32_t cols, void* stream) {
  HBA_REQUIRE(dst && src && rows > 0 && cols > 0, "hba_add_rows: bad arguments");
  add_rows_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      dst, ld_dst, dst_row_step < 1 ? 1 : dst_row_step, src, ld_src, rows, cols);
  return check_launch("hba_add_rows");
}

extern "C" int hba_nonfinite_flag(const float* x, int64_t n, int32_t* flag, void* stream) {
  HBA_REQUIRE(x && flag && n > 0, "hba_nonfinite_flag: bad arguments");
  nonfinite_flag_kernel<<<grid_for(n, 256, 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, n, flag);
  return check_launch("hba_nonfinite_flag");
}
