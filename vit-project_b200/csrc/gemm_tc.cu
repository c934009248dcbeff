// tcgen05 / TMEM / TMA GEMM for sm_100a:  C[M,N] = epilogue(A[M,K] . B[N,K]^T), bf16 in, fp32 acc.
//
// One persistent CTA per SM, CTAs paired into 2-CTA clusters (cta_group::2): a pair owns a
// 256 x BN tile of C.  10 warps per CTA, warp-specialised:
//   warp 0 (one lane)  TMA producer: its 128 rows of A and its BN/2 rows of B per k-block
//                      (SWIZZLE_128B boxes) into a 6-stage smem ring; bytes of both CTAs are
//                      accounted on the leader's mbarrier
//   warp 1 (one lane, leader CTA only)  tcgen05.mma.cta_group::2 issuer: 256 x BN x 16 UMMAs reading
//                      both CTAs' smem, accumulators in both CTAs' TMEM (128 rows each), 2 accumulator
//                      stages so that the epilogue of tile i overlaps the main loop of tile i+1;
//                      multicast tcgen05.commit frees the smem slot / publishes the tile in both CTAs
//   warps 2..9         epilogue: tcgen05.ld 32 lanes x 32 columns -> registers -> fused
//                      bias / QuickGELU / GELU / activation-gradient / residual -> global
// "fp32 mode" (nsplit == 3) runs three bf16 passes per k-block over hi/lo split operands
// (hi.hi + lo.hi + hi.lo), which reproduces fp32 products to ~2^-16 on the bf16 tensor pipe.
//
// Replaces F.linear at torch/nn/functional.py:6244 (in_proj), :6690 (out_proj) and the CLIP / timm
// MLP linears reached through the reference's CLIPHBA.forward (NEW:298) and VIT:138-140.
#include "common.cuh"

namespace hba {

constexpr int BM = 128;
constexpr int BK = 64;
// Epilogue geometry.  16 warps (four per TMEM lane quarter, each draining a quarter of the tile's
// columns in 32 x 16 chunks): the fused epilogues (GELU / GELU' / residual / two outputs) are issue- and
// latency-bound on the CUDA cores, and with 8 warps (2 per scheduler, 45 % issue utilisation) they, not
// the tensor pipe, set the tile time of every short-K GEMM (K = 768: 11 us epilogue vs 7 us main loop).
// 18 warps x 32 threads caps the kernel at 112 registers per thread; the 16-column chunk fits.
constexpr int kEpiWarps = 16;
constexpr int kChunkCols = 16;
constexpr int kGemmThreads = 64 + 32 * kEpiWarps;

// A CTA pair computes a 256 x BN tile, each CTA staging its own 128 rows of A and only HALF of the B
// tile -> 1/3 fewer bytes through the L2->SM fabric per FLOP than 128 x BN tiles (the fabric, not the
// tensor pipe, bounded a single-CTA kernel: 10.7 TB/s of TMA traffic at 44 % tensor-pipe utilisation,
// profiles/r01_gemm_attn_ncu_full.md)
template <int BN>
struct GemmCfg {
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = (BN / 2) * BK * 2;
  static constexpr int kStages = (192 * 1024) / (kABytes + kBBytes) > 8 ? 8 : (192 * 1024) / (kABytes + kBBytes);
  static constexpr int kTmemCols = 2 * BN;  // two accumulator stages
  static constexpr int kStagingBytes = kEpiWarps * 32 * kChunkCols * 4;  // per-warp transposition tiles of the epilogue
  static constexpr int kSmemBytes = kStages * (kABytes + kBBytes) + kStagingBytes + 1024 /*align*/ + 256 /*bars*/;
};

struct GemmArgs {
  int M, N, K;
  int nsplit, a_lo_off, b_lo_off;
  float alpha;
  const float* bias;
  const float* residual;
  int ldr;
  int act;
  const void* aux;
  int ld_aux, aux_dtype;
  void* pre_out;
  int ld_pre, pre_dtype;
  float* out_f32;
  int ld_f32;
  __nv_bfloat16* out_bf16;
  int ld_bf16, out_lo_off;
  int transpose_out;
  int a_mn, b_mn;  // operand stored MN-major: [K rows, M (resp. N) columns]
  float* colsum;   // optional [ceil(M / 32), N]: column sums of the bf16 output per 32-row group
  int k_slices;    // split-K: work item = (tile, K slice); slice s writes out_f32 + s * slice_stride
  size_t slice_stride;
  // tail splitting (k_slices == 1): tiles [tail_first, total) - the partial last round of the static schedule -
  // are cut into tail_f column slabs of BN / tail_f columns, one work item each, so that the last round keeps
  // ~all CTA pairs busy for 1 / tail_f of a tile time.  Every output element still accumulates its K products in
  // the same order: results are bit-identical to the unsplit schedule.
  int tail_first, tail_f;
};

// x * sigmoid(1.702 x) on the SFU fast paths (ex2.approx + rcp.approx, ~2 ulp): the epilogue of the
// c_fc GEMM evaluates this 33.7 M times per layer and must stay under the main loop's time
__device__ __forceinline__ float quickgelu(float v) {
  return __fdividef(v, 1.0f + __expf(-1.702f * v));
}
__device__ __forceinline__ float quickgelu_grad(float a) {
  const float s = __fdividef(1.0f, 1.0f + __expf(-1.702f * a));
  return s * (1.0f + 1.702f * a * (1.0f - s));
}
// erf-GELU (timm / nn.GELU default, VIT:283) and its derivative.  erf(|x|) = 1 - poly5(t) exp(-x^2),
// t = 1 / (1 + p |x|) (Abramowitz-Stegun 7.1.26, |error| <= 1.5e-7 = fp32 epsilon): one ex2.approx and
// one rcp.approx on the SFU plus 8 FMAs, and the exponential is the very one the derivative's
// density term needs.  erff() + expf() made the dX GEMM of fc2 epilogue-bound (858 us vs 250 us).
// h(v) = 0.5 * erfc(|v| / sqrt 2): Phi(v) = h for v < 0, 1 - h for v > 0.  `e` = exp(-v^2 / 2).
__device__ __forceinline__ float half_erfc_abs(float av, float e) {
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f * 0.70710678118654752f, av, 1.0f)));
  float p = fmaf(t, 0.5f * 1.061405429f, 0.5f * -1.453152027f);
  p = fmaf(p, t, 0.5f * 1.421413741f);
  p = fmaf(p, t, 0.5f * -0.284496736f);
  p = fmaf(p, t, 0.5f * 0.254829592f);
  return p * t * e;
}
__device__ __forceinline__ float exp_neg_half_sq(float v) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(v * v * -0.72134752044448170f));  // -0.5 * log2(e)
  return e;
}
// gelu(v) = v Phi(v) = relu(v) - |v| h(v)
__device__ __forceinline__ float gelu_erf(float v) {
  const float av = fabsf(v);
  return fmaf(-av, half_erfc_abs(av, exp_neg_half_sq(v)), fmaxf(v, 0.0f));
}
// gelu'(a) = Phi(a) + a phi(a)
__device__ __forceinline__ float gelu_erf_grad(float a) {
  const float e = exp_neg_half_sq(a);
  const float h = half_erfc_abs(fabsf(a), e);
  const float phi_cdf = a > 0.0f ? 1.0f - h : h;
  return fmaf(a * 0.39894228040143268f, e, phi_cdf);
}

// transposed store (C^T) for one thread: row `row`, 32 consecutive columns starting at `col`; for a
// fixed column the 32 lanes of the warp write 32 consecutive rows, i.e. contiguous memory.  Supports
// alpha and bias only (hba_gemm_bf16 rejects the other epilogue options with transpose_out).
__device__ __forceinline__ void epilogue_chunk_transposed(const GemmArgs& g, const uint32_t* r, int row,
                                                          int col) {
#pragma unroll
  for (int j = 0; j < kChunkCols; ++j) {
    if (col + j < g.N) {
      float v = __uint_as_float(r[j]) * g.alpha;
      if (g.bias) v += __ldg(g.bias + col + j);
      if (g.out_f32) g.out_f32[(size_t)(col + j) * g.ld_f32 + row] = v;
      if (g.out_bf16) {
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        g.out_bf16[(size_t)(col + j) * g.ld_bf16 + row] = h;
        if (g.out_lo_off > 0)
          g.out_bf16[(size_t)(col + j) * g.ld_bf16 + g.out_lo_off + row] =
              __float2bfloat16_rn(v - __bfloat162float(h));
      }
    }
  }
}

__device__ __forceinline__ void tmem_ld_chunk(uint32_t taddr, uint32_t* r) {
  static_assert(kChunkCols == 16 || kChunkCols == 32, "epilogue chunk is 16 or 32 columns");
  if constexpr (kChunkCols == 32) {
    tmem_ld_32x32b_x32(taddr, r);
  } else {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
  }
}

// ---- coalesced epilogue --------------------------------------------------------------------
// tcgen05.ld hands every thread one accumulator ROW (32 columns); storing that directly makes every
// warp-wide store touch 32 different lines, 16 bytes each.  The chunk is therefore transposed through
// a per-warp 4 KB shared-memory tile (16-byte granules XOR-swizzled by the row: conflict-free both
// ways); afterwards lane l owns the float4 at columns 4*(l&7).. of rows 4*i + (l>>3), i = 0..7, so a
// warp-wide access covers 4 rows x 128 contiguous bytes.  Bias, activation, activation gradient,
// residual and every output (fp32 / bf16 hi[/lo] / pre-activation) use that layout.
struct Vec4 {
  float x[4];
};
// explicit shared-space accesses (the 1024-byte aligned base is computed through an integer, which
// would otherwise demote these to generic LD/ST)
__device__ __forceinline__ void sts128(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(addr)
               : "memory");
  return v;
}
__device__ __forceinline__ Vec4 ld4_f32(const float* p) {
  const float4 t = __ldg(reinterpret_cast<const float4*>(p));
  return Vec4{{t.x, t.y, t.z, t.w}};
}
__device__ __forceinline__ Vec4 ld4_bf16(const __nv_bfloat16* p) {
  const uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
  const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&t.x);
  const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&t.y);
  return Vec4{{__low2float(a), __high2float(a), __low2float(b), __high2float(b)}};
}
__device__ __forceinline__ void st4_f32(float* p, const Vec4& v) {
  *reinterpret_cast<float4*>(p) = make_float4(v.x[0], v.x[1], v.x[2], v.x[3]);
}
__device__ __forceinline__ void st4_bf16(__nv_bfloat16* p, const Vec4& v) {
  *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16x2(v.x[0], v.x[1]), pack_bf16x2(v.x[2], v.x[3]));
}

__device__ __forceinline__ float act_runtime(int act, float v, float a) {
  switch (act) {
    case HBA_ACT_QUICKGELU: return quickgelu(v);
    case HBA_ACT_GELU_ERF: return gelu_erf(v);
    case HBA_ACT_QUICKGELU_GRAD: return v * quickgelu_grad(a);
    case HBA_ACT_GELU_ERF_GRAD: return v * gelu_erf_grad(a);
    default: return v;
  }
}

// one 32-row x CC-column chunk of the tile (CC = kChunkCols); `r` = this thread's accumulator row
// (lane = row), `stage` = shared-space address of this warp's private staging tile (32 rows x CC fp32).
// ACT is a template parameter: each kernel instance carries only its own activation code (the erf
// variants are long and a kernel with all five thrashed the instruction cache).
// After the transposition lane l owns the float4 at columns 4*(l % LPR) of rows RPA*i + l / LPR.
template <int ACT>
__device__ __forceinline__ void epilogue_chunk_coalesced(const GemmArgs& g, float* __restrict__ out_f32,
                                                         const uint32_t* r, uint32_t stage, int row0,
                                                         int col0, int lane) {
  constexpr int CC = kChunkCols;
  constexpr int LPR = CC / 4;       // lanes (float4 granules) per row
  constexpr int RPA = 32 / LPR;     // rows covered by one warp-wide access
  constexpr int NI = 32 / RPA;      // accesses per chunk
  // 16-byte granule XOR swizzle by the row: conflict-free for the row-per-lane writes and the
  // RPA-rows-per-access reads (LPR = 8: row & 7;  LPR = 4: (row >> 1) & 3, rows are 64 B apart)
  auto swz = [](int row) { return LPR == 8 ? (row & 7) : ((row >> 1) & 3); };
  const int cq = lane % LPR, rsub = lane / LPR;
  const int col = col0 + 4 * cq;
  const int nvalid = g.N - col;  // >= 4: the whole float4 is in range
  const bool vec = nvalid >= 4;
  // lanes that take the vector path: in a chunk that N cuts (N % 16 != 0) the lanes of the columns past N
  // do not, and the column-sum shuffles below must name only the lanes that execute them
  const unsigned vec_lanes = g.colsum ? __ballot_sync(0xffffffffu, vec) : 0u;
  constexpr bool kGrad = (ACT == HBA_ACT_QUICKGELU_GRAD || ACT == HBA_ACT_GELU_ERF_GRAD);
  // loads that do not depend on the accumulator are issued first (they overlap the transposition)
  Vec4 bias = {{0.f, 0.f, 0.f, 0.f}};
  Vec4 res[NI];
  Vec4 aux[kGrad ? NI : 1];
  if (vec) {
    if (g.bias) bias = ld4_f32(g.bias + col);
    if constexpr (kGrad) {
      // all pre-activation vectors of the chunk in flight at once (one after the other inside the math
      // loop they cost one exposed DRAM round trip each: 785 us for the fc2 dX GEMM of ViT-B/16)
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const int row = min(row0 + RPA * i + rsub, g.M - 1);
        if (g.aux_dtype == HBA_DT_F32) {
          const float* p = static_cast<const float*>(g.aux) + (size_t)row * g.ld_aux + col;
          if ((g.ld_aux & 3) == 0) aux[i] = ld4_f32(p);
          else aux[i] = Vec4{{__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3)}};
        } else {
          const __nv_bfloat16* p = static_cast<const __nv_bfloat16*>(g.aux) + (size_t)row * g.ld_aux + col;
          if ((g.ld_aux & 3) == 0) aux[i] = ld4_bf16(p);
          else aux[i] = Vec4{{__bfloat162float(p[0]), __bfloat162float(p[1]), __bfloat162float(p[2]),
                              __bfloat162float(p[3])}};
        }
      }
    }
    if (g.residual) {
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const int row = row0 + RPA * i + rsub;
        res[i] = Vec4{{0.f, 0.f, 0.f, 0.f}};
        if (row < g.M) res[i] = ld4_f32(g.residual + (size_t)row * g.ldr + col);
      }
    }
  }
  if (g.alpha == 1.0f) {
#pragma unroll
    for (int j = 0; j < LPR; ++j)
      sts128(stage + 16u * (lane * LPR + (j ^ swz(lane))), __uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
             __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
  } else {
#pragma unroll
    for (int j = 0; j < LPR; ++j)
      sts128(stage + 16u * (lane * LPR + (j ^ swz(lane))), __uint_as_float(r[4 * j]) * g.alpha,
             __uint_as_float(r[4 * j + 1]) * g.alpha, __uint_as_float(r[4 * j + 2]) * g.alpha,
             __uint_as_float(r[4 * j + 3]) * g.alpha);
  }
  __syncwarp();
  if (vec) {
    Vec4 v[NI];
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int rl = RPA * i + rsub;
      const float4 t = lds128(stage + 16u * (rl * LPR + (cq ^ swz(rl))));
      v[i] = Vec4{{t.x + bias.x[0], t.y + bias.x[1], t.z + bias.x[2], t.w + bias.x[3]}};
    }
    if (g.pre_out) {
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const int row = row0 + RPA * i + rsub;
        if (row >= g.M) continue;
        if (g.pre_dtype == HBA_DT_F32)
          st4_f32(static_cast<float*>(g.pre_out) + (size_t)row * g.ld_pre + col, v[i]);
        else
          st4_bf16(static_cast<__nv_bfloat16*>(g.pre_out) + (size_t)row * g.ld_pre + col, v[i]);
      }
    }
    if constexpr (ACT == HBA_ACT_QUICKGELU) {
#pragma unroll
      for (int i = 0; i < NI; ++i)
#pragma unroll
        for (int e = 0; e < 4; ++e) v[i].x[e] = quickgelu(v[i].x[e]);
    } else if constexpr (ACT == HBA_ACT_GELU_ERF) {
#pragma unroll
      for (int i = 0; i < NI; ++i)
#pragma unroll
        for (int e = 0; e < 4; ++e) v[i].x[e] = gelu_erf(v[i].x[e]);
    } else if constexpr (kGrad) {
#pragma unroll
      for (int i = 0; i < NI; ++i)
#pragma unroll
        for (int e = 0; e < 4; ++e)
          v[i].x[e] *= (ACT == HBA_ACT_QUICKGELU_GRAD) ? quickgelu_grad(aux[i].x[e]) : gelu_erf_grad(aux[i].x[e]);
    }
    if (g.residual) {
#pragma unroll
      for (int i = 0; i < NI; ++i)
#pragma unroll
        for (int e = 0; e < 4; ++e) v[i].x[e] += res[i].x[e];
    }
    if (out_f32) {
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const int row = row0 + RPA * i + rsub;
        if (row < g.M) st4_f32(out_f32 + (size_t)row * g.ld_f32 + col, v[i]);
      }
    }
    if (g.colsum) {
      // bias gradient fused into the GEMM that produces dY: column sums of the bf16-rounded outputs of
      // this 32-row x CC-column chunk; every (row group, column) is written by exactly one warp, the
      // row groups are summed afterwards in a fixed order (hba_colsum) - deterministic
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        if (row0 + RPA * i + rsub < g.M) {
          s0 += __bfloat162float(__float2bfloat16_rn(v[i].x[0]));
          s1 += __bfloat162float(__float2bfloat16_rn(v[i].x[1]));
          s2 += __bfloat162float(__float2bfloat16_rn(v[i].x[2]));
          s3 += __bfloat162float(__float2bfloat16_rn(v[i].x[3]));
        }
      }
#pragma unroll
      for (int o = LPR; o < 32; o <<= 1) {   // (lane ^ o keeps the column granule cq: vec_lanes holds both)
        s0 += __shfl_xor_sync(vec_lanes, s0, o);
        s1 += __shfl_xor_sync(vec_lanes, s1, o);
        s2 += __shfl_xor_sync(vec_lanes, s2, o);
        s3 += __shfl_xor_sync(vec_lanes, s3, o);
      }
      if (rsub == 0)
        *reinterpret_cast<float4*>(g.colsum + (size_t)(row0 >> 5) * g.N + col) = make_float4(s0, s1, s2, s3);
    }
    if (g.out_bf16) {
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const int row = row0 + RPA * i + rsub;
        if (row >= g.M) continue;
        __nv_bfloat16* p = g.out_bf16 + (size_t)row * g.ld_bf16 + col;
        st4_bf16(p, v[i]);
        if (g.out_lo_off > 0) {
          Vec4 l;
#pragma unroll
          for (int e = 0; e < 4; ++e)
            l.x[e] = v[i].x[e] - __bfloat162float(__float2bfloat16_rn(v[i].x[e]));
          st4_bf16(p + g.out_lo_off, l);
        }
      }
    }
  } else if (nvalid > 0) {
    // ragged last columns (N % 4 != 0): element-wise, not unrolled (cold path)
#pragma unroll 1
    for (int i = 0; i < NI; ++i) {
      const int rl = RPA * i + rsub;
      const int row = row0 + rl;
      if (row >= g.M) continue;
      const float4 t = lds128(stage + 16u * (rl * LPR + (cq ^ swz(rl))));
      const float tv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll 1
      for (int e = 0; e < nvalid; ++e) {
        float v = tv[e] + (g.bias ? __ldg(g.bias + col + e) : 0.f);
        if (g.pre_out) {
          if (g.pre_dtype == HBA_DT_F32)
            static_cast<float*>(g.pre_out)[(size_t)row * g.ld_pre + col + e] = v;
          else
            static_cast<__nv_bfloat16*>(g.pre_out)[(size_t)row * g.ld_pre + col + e] = __float2bfloat16_rn(v);
        }
        float a = 0.f;
        if (kGrad)
          a = g.aux_dtype == HBA_DT_F32
                  ? __ldg(static_cast<const float*>(g.aux) + (size_t)row * g.ld_aux + col + e)
                  : __bfloat162float(static_cast<const __nv_bfloat16*>(g.aux)[(size_t)row * g.ld_aux + col + e]);
        v = act_runtime(ACT, v, a);
        if (g.residual) v += __ldg(g.residual + (size_t)row * g.ldr + col + e);
        if (out_f32) out_f32[(size_t)row * g.ld_f32 + col + e] = v;
        if (g.out_bf16) {
          const __nv_bfloat16 h = __float2bfloat16_rn(v);
          g.out_bf16[(size_t)row * g.ld_bf16 + col + e] = h;
          if (g.out_lo_off > 0)
            g.out_bf16[(size_t)row * g.ld_bf16 + g.out_lo_off + col + e] =
                __float2bfloat16_rn(v - __bfloat162float(h));
        }
      }
    }
  }
  __syncwarp();  // the staging tile is rewritten by the next chunk
}

// work item -> (tile, K slice, first column inside the tile, width in columns)
struct GemmItem {
  int tile, slice, n_off, bn;
};
template <int BN>
__device__ __forceinline__ GemmItem decode_item(const GemmArgs& g, int item, int total_tiles) {
  GemmItem it;
  if (g.tail_f > 1 && item >= g.tail_first) {
    const int idx = item - g.tail_first;
    it.bn = BN / g.tail_f;
    it.tile = g.tail_first + idx / g.tail_f;
    it.n_off = (idx % g.tail_f) * it.bn;
    it.slice = 0;
  } else {
    it.tile = item % total_tiles, it.slice = item / total_tiles, it.n_off = 0, it.bn = BN;
  }
  return it;
}

template <int BN, int ACT>
__global__ void __launch_bounds__(kGemmThreads, 1)
    gemm_tc_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                   const __grid_constant__ CUtensorMap tma_b2, const __grid_constant__ CUtensorMap tma_b4,
                   const GemmArgs g) {
  using Cfg = GemmCfg<BN>;
  constexpr int kStages = Cfg::kStages;
  constexpr int BNC = BN / 2;   // rows of B this CTA stages per k-block
  constexpr int TM = 2 * BM;    // rows of C per tile (per CTA pair)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* sA = smem;
  uint8_t* sB = sA + kStages * Cfg::kABytes;
  uint8_t* sStage = sB + kStages * Cfg::kBBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sB + kStages * Cfg::kBBytes + Cfg::kStagingBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tfull_bar = empty_bar + kStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  // broadcast from lane 0: the compiler then knows the role branches below are warp-uniform and keeps
  // descriptors / barrier addresses in uniform registers (no per-instruction waterfall loops around
  // UTCHMMA / UTMALDG)
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();  // 0 = leader (issues the UMMAs)
  const int worker = blockIdx.x / 2, num_workers = gridDim.x / 2;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);   // the leader's producer arrives (+ the tx bytes of both CTAs)
      mbar_init(&empty_bar[i], 1);  // one (multicast) tcgen05.commit
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], kEpiWarps * 2);  // one arrival per epilogue warp of the pair
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc_pair(tmem_slot, Cfg::kTmemCols);
  tc_fence_before();
  cluster_sync_all();  // the peer's barriers must be live before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int num_m_tiles = (g.M + TM - 1) / TM;
  const int num_n_tiles = (g.N + BN - 1) / BN;
  const int total_tiles = num_m_tiles * num_n_tiles;
  const int kblocks = (g.K + BK - 1) / BK;  // a ragged last block is zero-filled by TMA
  // split-K: item = slice * total_tiles + tile; slice s covers k-blocks [s * kb_per, min(.., kblocks))
  const int total_items = g.tail_f > 1 ? g.tail_first + (total_tiles - g.tail_first) * g.tail_f
                                        : total_tiles * g.k_slices;
  const int kb_per = (kblocks + g.k_slices - 1) / g.k_slices;

  if (warp == 0) {
    {
      int stage = 0;
      uint32_t phase = 0;
      // where this CTA's TMA bytes are accounted: the pair leader's barriers
      const uint32_t full0 = mapa_u32(&full_bar[0], 0);
      for (int item = worker; item < total_items; item += num_workers) {
        const GemmItem wi = decode_item<BN>(g, item, total_tiles);
        const int tile = wi.tile, slice = wi.slice;
        const int bnc = wi.bn / 2;   // rows of B this CTA stages for the item
        const int m0 = (tile / num_n_tiles) * TM + rank * BM;
        const int n0 = (tile % num_n_tiles) * BN + wi.n_off + rank * bnc;
        const CUtensorMap* tmb = wi.bn == BN ? &tma_b : (wi.bn * 2 == BN ? &tma_b2 : &tma_b4);
        const uint32_t stage_bytes = (uint32_t)(2 * (Cfg::kABytes + bnc * BK * 2));
        const int kb_end = min(kblocks, (slice + 1) * kb_per);
        for (int kb = slice * kb_per; kb < kb_end; ++kb) {
          for (int s = 0; s < g.nsplit; ++s) {
            const int a_col = kb * BK + (s == 1 ? g.a_lo_off : 0);
            const int b_col = kb * BK + (s == 2 ? g.b_lo_off : 0);
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* dA = sA + stage * Cfg::kABytes;
            uint8_t* dB = sB + stage * Cfg::kBBytes;
            const uint32_t fb = full0 + 8u * stage;
            if (elect_one()) {
            if (rank == 0)
              mbar_arrive_expect_tx(&full_bar[stage], stage_bytes);
            if (!g.a_mn) {
              tma_load_2d_pair(dA, &tma_a, fb, a_col, m0);
            } else {  // [K, M] storage: BM/64 boxes of 64 k-rows x 64 m-columns, 8 KB apart (LBO)
#pragma unroll
              for (int j = 0; j < BM / 64; ++j)
                tma_load_2d_pair(dA + j * 8192, &tma_a, fb, m0 + 64 * j + (s == 1 ? g.a_lo_off : 0),
                                 kb * BK);
            }
            if (!g.b_mn) {
              tma_load_2d_pair(dB, tmb, fb, b_col, n0);
            } else {
#pragma unroll
              for (int j = 0; j < BNC / 64; ++j)
                tma_load_2d_pair(dB + j * 8192, &tma_b, fb, n0 + 64 * j + (s == 2 ? g.b_lo_off : 0),
                                 kb * BK);
            }
            }
            __syncwarp();
            if (++stage == kStages) stage = 0, phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      const uint32_t idesc_flags = (g.a_mn ? (1u << 15) : 0u) | (g.b_mn ? (1u << 16) : 0u);
      // K-major: +32 B per 16-element k-step inside the 128-byte swizzle row (start address += 2);
      // MN-major: 16 k-rows of 128 B further down (start address += 128)
      const uint32_t a_step = g.a_mn ? 128u : 2u, b_step = g.b_mn ? 128u : 2u;
      const uint64_t mn_lbo = (uint64_t)(8192 >> 4) << 16;  // next 64-wide MN block of an MN-major tile
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int item = worker; item < total_items; item += num_workers) {
        const GemmItem wi = decode_item<BN>(g, item, total_tiles);
        const int slice = wi.slice;
        const uint32_t idesc = make_idesc_bf16(TM, wi.bn) | idesc_flags;
        const int kiters = (min(kblocks, (slice + 1) * kb_per) - slice * kb_per) * g.nsplit;
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int it = 0; it < kiters; ++it) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          uint64_t a_desc = make_smem_desc_sw128(smem_u32(sA + stage * Cfg::kABytes));
          uint64_t b_desc = make_smem_desc_sw128(smem_u32(sB + stage * Cfg::kBBytes));
          if (g.a_mn) a_desc = (a_desc & ~((uint64_t)0x3FFF << 16)) | mn_lbo;
          if (g.b_mn) b_desc = (b_desc & ~((uint64_t)0x3FFF << 16)) | mn_lbo;
          if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint32_t accum = (it > 0 || k > 0) ? 1u : 0u;
            umma_bf16_pair(d_tmem, a_desc + a_step * k, b_desc + b_step * k, idesc, accum);
          }
          // frees the smem slot (in both CTAs of the pair) once these MMAs have read it
          umma_commit_pair(&empty_bar[stage], 3);
          if (it == kiters - 1) umma_commit_pair(&tfull_bar[acc], 3);
          }
          __syncwarp();
          if (++stage == kStages) stage = 0, phase ^= 1;
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else {
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int part = (warp - 2) >> 2;  // which 1 / (kEpiWarps / 4) of the tile's columns this warp drains
    constexpr int kParts = kEpiWarps / 4;
    const uint32_t tempty_addr[2] = {mapa_u32(&tempty_bar[0], 0), mapa_u32(&tempty_bar[1], 0)};
    int acc = 0;
    uint32_t acc_phase = 0;
    // The epilogue's own inputs (residual / pre-activation rows of this warp's half tile) are pulled
    // into L2 one work item ahead: when the epilogue is the longer stage the accumulator is already
    // waiting, and loads issued only then paid a full DRAM round trip per 32 x 32 chunk.
    auto prefetch_inputs = [&](int it) {
      if (it >= total_items || g.transpose_out || (!g.residual && !g.aux)) return;
      const GemmItem pi = decode_item<BN>(g, it, total_tiles);
      const int tl = pi.tile, pw = pi.bn / kParts;   // this warp's column share of the item
      const int prow = (tl / num_n_tiles) * TM + rank * BM + q * 32 + lane;
      if (prow >= g.M) return;
      const int c0 = (tl % num_n_tiles) * BN + pi.n_off + part * pw;
      if (g.residual) {
        const char* p = reinterpret_cast<const char*>(g.residual + (size_t)prow * g.ldr + c0);
        for (int b = 0; b < pw * 4; b += 128)
          if (c0 + b / 4 < g.N) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + b));
      }
      if (g.aux) {
        const int esz = g.aux_dtype == HBA_DT_F32 ? 4 : 2;
        const char* p = static_cast<const char*>(g.aux) + ((size_t)prow * g.ld_aux + c0) * esz;
        for (int b = 0; b < pw * esz; b += 128)
          if (c0 + b / esz < g.N) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + b));
      }
    };
    prefetch_inputs(worker);
    for (int item = worker; item < total_items; item += num_workers) {
      const GemmItem wi = decode_item<BN>(g, item, total_tiles);
      const int tile = wi.tile, slice = wi.slice;
      const int chunks_per_warp = wi.bn / kChunkCols / kParts;   // BN / tail_f >= 64 columns: at least one chunk
      const int m0 = (tile / num_n_tiles) * TM + rank * BM;
      const int n0 = (tile % num_n_tiles) * BN + wi.n_off;
      const int row = m0 + q * 32 + lane;
      float* const out_f32 = g.out_f32 ? g.out_f32 + (size_t)slice * g.slice_stride : nullptr;
      prefetch_inputs(item + num_workers);
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
#pragma unroll 1
      for (int c = part * chunks_per_warp; c < (part + 1) * chunks_per_warp; ++c) {
        uint32_t r[kChunkCols];
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN + c * kChunkCols;
        tmem_ld_chunk(taddr, r);
        tmem_ld_wait();
        const int col = n0 + c * kChunkCols;
        if (g.transpose_out) {
          if (row < g.M && col < g.N) epilogue_chunk_transposed(g, r, row, col);
        } else if (m0 + q * 32 < g.M && col < g.N) {  // warp-uniform
          epilogue_chunk_coalesced<ACT>(g, out_f32, r, smem_u32(sStage) + (warp - 2) * (32 * kChunkCols * 4), m0 + q * 32, col, lane);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty_addr[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }
  tc_fence_before();
  cluster_sync_relaxed();  // the leader's UMMAs read the peer's smem and signal its barriers until the end
  if (warp == 1) tmem_dealloc_pair(tmem_base, Cfg::kTmemCols);
}

// out[r, c] = epilogue(sum_s part[s][r, c])  (split-K reduction, fixed order: deterministic).  The epilogue is
// the GEMM's own (bias -> pre-activation output -> activation / activation gradient -> residual -> fp32 / bf16
// hi[/lo] outputs): skinny problems (the CLS / EOT row GEMMs, M = 32 / 66: 3..16 output tiles for 74 CTA pairs,
// each streaming the whole K extent of its weight columns through ONE SM pair) are split along K so that the weight
// matrix is pulled by many SMs at once, and finished here.
struct ReduceArgs {
  const float* part;
  size_t slice_stride;
  int slices, rows, cols, ld;
  const float* bias;
  const float* residual;
  int ldr;
  int act;
  const void* aux;
  int ld_aux, aux_dtype;
  void* pre_out;
  int ld_pre, pre_dtype;
  float* out_f32;
  int ld_f32;
  __nv_bfloat16* out_bf16;
  int ld_bf16, out_lo_off;
};

__global__ void __launch_bounds__(256) splitk_reduce_kernel(const ReduceArgs a) {
  const int c4 = a.cols >> 2;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)a.rows * c4;
       i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / c4), c = (int)(i % c4) * 4;
    float4 acc = *reinterpret_cast<const float4*>(a.part + (size_t)r * a.ld + c);
    for (int s = 1; s < a.slices; ++s) {
      const float4 v = *reinterpret_cast<const float4*>(a.part + s * a.slice_stride + (size_t)r * a.ld + c);
      acc.x += v.x, acc.y += v.y, acc.z += v.z, acc.w += v.w;
    }
    Vec4 v = {{acc.x, acc.y, acc.z, acc.w}};
    if (a.bias) {
      const Vec4 b = ld4_f32(a.bias + c);
#pragma unroll
      for (int e = 0; e < 4; ++e) v.x[e] += b.x[e];
    }
    if (a.pre_out) {
      if (a.pre_dtype == HBA_DT_F32) st4_f32(static_cast<float*>(a.pre_out) + (size_t)r * a.ld_pre + c, v);
      else st4_bf16(static_cast<__nv_bfloat16*>(a.pre_out) + (size_t)r * a.ld_pre + c, v);
    }
    if (a.act != HBA_ACT_NONE) {
      Vec4 x = {{0.f, 0.f, 0.f, 0.f}};
      if (a.aux) {
        if (a.aux_dtype == HBA_DT_F32) {
          const float* p = static_cast<const float*>(a.aux) + (size_t)r * a.ld_aux + c;
          x = Vec4{{__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3)}};
        } else {
          const __nv_bfloat16* p = static_cast<const __nv_bfloat16*>(a.aux) + (size_t)r * a.ld_aux + c;
          x = Vec4{{__bfloat162float(p[0]), __bfloat162float(p[1]), __bfloat162float(p[2]), __bfloat162float(p[3])}};
        }
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) v.x[e] = act_runtime(a.act, v.x[e], x.x[e]);
    }
    if (a.residual) {
      const Vec4 q = ld4_f32(a.residual + (size_t)r * a.ldr + c);
#pragma unroll
      for (int e = 0; e < 4; ++e) v.x[e] += q.x[e];
    }
    if (a.out_f32) st4_f32(a.out_f32 + (size_t)r * a.ld_f32 + c, v);
    if (a.out_bf16) {
      __nv_bfloat16* p = a.out_bf16 + (size_t)r * a.ld_bf16 + c;
      st4_bf16(p, v);
      if (a.out_lo_off > 0) {
        Vec4 l;
#pragma unroll
        for (int e = 0; e < 4; ++e) l.x[e] = v.x[e] - __bfloat162float(__float2bfloat16_rn(v.x[e]));
        st4_bf16(p + a.out_lo_off, l);
      }
    }
  }
}

// Encoding a CUtensorMap costs ~1 us of host time (cuTensorMapEncodeTiled) and every GEMM launch needs two; the
// operands of a training step are the same few hundred (pointer, shape, stride, box) tuples step after step, so
// the encoded descriptors are kept in a small direct-mapped, per-thread cache.  A descriptor depends on nothing but
// those six numbers (no device or context state), so a stale entry is impossible: equal key = equal descriptor.
struct TmaKey {
  const void* ptr;
  uint64_t rows, cols, ld;
  uint32_t box_rows, box_cols;
  bool operator==(const TmaKey& o) const {
    return ptr == o.ptr && rows == o.rows && cols == o.cols && ld == o.ld && box_rows == o.box_rows &&
           box_cols == o.box_cols;
  }
};
static int cached_tma_2d_bf16(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld,
                              uint32_t box_rows, uint32_t box_cols) {
  constexpr int kSlots = 1024;
  struct Slot {
    TmaKey key;
    CUtensorMap map;
    bool valid;
  };
  static thread_local Slot* slots = nullptr;
  if (!slots) slots = new Slot[kSlots]();
  const TmaKey key{ptr, rows, cols, ld, box_rows, box_cols};
  uint64_t h = (uint64_t)(uintptr_t)ptr * 0x9E3779B97F4A7C15ull;
  h ^= (rows * 0xC2B2AE3D27D4EB4Full) ^ (cols << 21) ^ (ld << 7) ^ ((uint64_t)box_rows << 40) ^ box_cols;
  Slot& sl = slots[(h >> 32) % kSlots];
  if (sl.valid && sl.key == key) {
    *map = sl.map;
    return HBA_OK;
  }
  HBA_CHECK(make_tma_2d_bf16(map, ptr, rows, cols, ld, box_rows, box_cols));
  sl.key = key, sl.map = *map, sl.valid = true;
  return HBA_OK;
}

template <int BN, int ACT>
static int launch_gemm(const hba_gemm_params* p, const GemmArgs& g, cudaStream_t stream) {
  using Cfg = GemmCfg<BN>;
  static SmemAttr smem_attr;
  HBA_CHECK(ensure_dyn_smem(gemm_tc_kernel<BN, ACT>, Cfg::kSmemBytes, smem_attr, "gemm_tc_kernel"));
  constexpr int BNC = BN / 2;
  const uint64_t a_cols = (uint64_t)p->K + (p->nsplit == 3 ? (uint64_t)p->a_lo_off : 0);
  const uint64_t b_cols = (uint64_t)p->K + (p->nsplit == 3 ? (uint64_t)p->b_lo_off : 0);
  CUtensorMap ta, tb;
  if (!p->a_mn_major) {
    HBA_CHECK(cached_tma_2d_bf16(&ta, p->A, p->M, a_cols, p->lda, BM, BK));
  } else {
    const uint64_t cols = (uint64_t)p->M + (p->nsplit == 3 ? (uint64_t)p->a_lo_off : 0);
    HBA_CHECK(cached_tma_2d_bf16(&ta, p->A, p->K, cols, p->lda, 64, 64));
  }
  if (!p->b_mn_major) {
    HBA_CHECK(cached_tma_2d_bf16(&tb, p->B, p->N, b_cols, p->ldb, BNC, BK));
  } else {
    const uint64_t cols = (uint64_t)p->N + (p->nsplit == 3 ? (uint64_t)p->b_lo_off : 0);
    HBA_CHECK(cached_tma_2d_bf16(&tb, p->B, p->K, cols, p->ldb, 64, 64));
  }
  const int tiles = ((p->M + 2 * BM - 1) / (2 * BM)) * ((p->N + BN - 1) / BN);
  int workers = num_sms() / 2;  // CTA pairs
  if (p->max_ctas > 0 && p->max_ctas / 2 < workers) workers = p->max_ctas / 2 > 0 ? p->max_ctas / 2 : 1;
  if (tiles * g.k_slices < workers) workers = tiles * g.k_slices;
  // tail splitting: cut the tiles of a partial last round into 2 or 4 column slabs when that shortens the round.
  // Slab times relative to a full tile (the kernel is bound by the bytes an SM takes in per k-block: its 16 KB of A
  // are re-read per slab, only the B share shrinks: (16 + 16 / f) / 32 -> 0.75 / 0.625; measured: the qkv GEMM
  // 8224 x 3072 x 1024 44.2 -> 42.7 us with f = 2, 5082 x 3072 x 768 36.4 -> 33.3 us with f = 4).
  GemmArgs ga = g;
  ga.tail_first = tiles, ga.tail_f = 1;
  CUtensorMap tb2 = tb, tb4 = tb;
  if (BN == 256 && g.k_slices == 1 && !p->a_mn_major && !p->b_mn_major && tiles > workers &&
      tiles % workers != 0) {
    const int rem = tiles % workers;
    const double cost1 = 1.0;
    const double cost2 = ((rem * 2 + workers - 1) / workers) * 0.75;
    const double cost4 = ((rem * 4 + workers - 1) / workers) * 0.65;
    int f = 1;
    if (cost2 < cost1 - 0.05 && cost2 <= cost4) f = 2;
    else if (cost4 < cost1 - 0.05) f = 4;
    if (f > 1) {
      ga.tail_first = tiles - rem, ga.tail_f = f;
      HBA_CHECK(cached_tma_2d_bf16(&tb2, p->B, p->N, b_cols, p->ldb, BNC / 2, BK));
      HBA_CHECK(cached_tma_2d_bf16(&tb4, p->B, p->N, b_cols, p->ldb, BNC / 4, BK));
    }
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(workers * 2));
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, ACT>, ta, tb, tb2, tb4, ga);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("gemm_tc_kernel<%d> launch: %s", BN, cudaGetErrorString(e));
    return HBA_ERR_CUDA;
  }
  return check_launch("gemm_tc_kernel");
}

}  // namespace hba

extern "C" int hba_gemm_bf16(const hba_gemm_params* p, void* stream) {
  using namespace hba;
  HBA_REQUIRE(p != nullptr, "hba_gemm_bf16: null params");
  HBA_REQUIRE(p->A && p->B, "hba_gemm_bf16: null operand");
  HBA_REQUIRE(p->M > 0 && p->N > 0 && p->K > 0, "hba_gemm_bf16: empty problem M=%d N=%d K=%d",
              p->M, p->N, p->K);
  // a ragged last k-block is zero-filled by TMA; a split K-major operand must then keep its hi part
  // zero padded up to the lo part (checked below through the lo offsets)
  HBA_REQUIRE(p->lda % 8 == 0 && p->ldb % 8 == 0, "hba_gemm_bf16: lda/ldb must be multiples of 8");
  HBA_REQUIRE(p->nsplit == 1 || p->nsplit == 3, "hba_gemm_bf16: nsplit must be 1 or 3");
  if (p->nsplit == 3)
    HBA_REQUIRE(p->a_lo_off >= (p->a_mn_major ? p->M : (p->K + BK - 1) / BK * BK) &&
                    p->b_lo_off >= (p->b_mn_major ? p->N : (p->K + BK - 1) / BK * BK) && p->a_lo_off % 8 == 0 &&
                    p->b_lo_off % 8 == 0,
                "hba_gemm_bf16: lo offsets must lie behind the hi part and be multiples of 8");
  HBA_REQUIRE(p->out_f32 || p->out_bf16 || p->pre_out, "hba_gemm_bf16: no output");
  HBA_REQUIRE(p->act >= HBA_ACT_NONE && p->act <= HBA_ACT_GELU_ERF_GRAD, "hba_gemm_bf16: bad act");
  if (p->act == HBA_ACT_QUICKGELU_GRAD || p->act == HBA_ACT_GELU_ERF_GRAD) {
    HBA_REQUIRE(p->aux != nullptr, "hba_gemm_bf16: activation gradient needs aux");
    // with ld_aux % 4 == 0 the epilogue loads aux four elements at a time (float4 / 8-byte bf16 vectors)
    HBA_REQUIRE(p->ld_aux % 4 != 0 || ((uintptr_t)p->aux & (p->aux_dtype == HBA_DT_F32 ? 15 : 7)) == 0,
                "hba_gemm_bf16: aux with ld %% 4 == 0 must be 16-byte (f32) / 8-byte (bf16) aligned");
  }
  if (p->transpose_out)
    HBA_REQUIRE(p->act == HBA_ACT_NONE && !p->residual && !p->pre_out,
                "hba_gemm_bf16: transpose_out supports alpha and bias only");
  if (!p->transpose_out) {
    HBA_REQUIRE(!p->out_f32 || (p->ld_f32 % 4 == 0 && ((uintptr_t)p->out_f32 & 15) == 0),
                "hba_gemm_bf16: out_f32 must be 16-byte aligned with ld %% 4 == 0");
    HBA_REQUIRE(!p->out_bf16 || (p->ld_bf16 % 8 == 0 && p->out_lo_off % 8 == 0 &&
                                 ((uintptr_t)p->out_bf16 & 15) == 0),
                "hba_gemm_bf16: out_bf16 must be 16-byte aligned with ld %% 8 == 0");
  }
  HBA_REQUIRE(!p->residual || (p->ldr % 4 == 0 && ((uintptr_t)p->residual & 15) == 0),
              "hba_gemm_bf16: residual must be 16-byte aligned with ld %% 4 == 0");
  HBA_REQUIRE(!p->bias || ((uintptr_t)p->bias & 15) == 0, "hba_gemm_bf16: bias must be 16-byte aligned");
  if (p->pre_out)
    HBA_REQUIRE(((uintptr_t)p->pre_out & 15) == 0 && p->ld_pre % 8 == 0,
                "hba_gemm_bf16: pre_out must be 16-byte aligned with ld %% 8 == 0");
  GemmArgs g;
  g.M = p->M, g.N = p->N, g.K = p->K;
  g.nsplit = p->nsplit, g.a_lo_off = p->a_lo_off, g.b_lo_off = p->b_lo_off;
  g.alpha = p->alpha;
  g.bias = p->bias, g.residual = p->residual, g.ldr = p->ldr;
  g.act = p->act, g.aux = p->aux, g.ld_aux = p->ld_aux, g.aux_dtype = p->aux_dtype;
  g.pre_out = p->pre_out, g.ld_pre = p->ld_pre, g.pre_dtype = p->pre_dtype;
  g.out_f32 = p->out_f32, g.ld_f32 = p->ld_f32;
  g.out_bf16 = static_cast<__nv_bfloat16*>(p->out_bf16), g.ld_bf16 = p->ld_bf16;
  g.out_lo_off = p->out_lo_off, g.transpose_out = p->transpose_out;
  g.a_mn = p->a_mn_major, g.b_mn = p->b_mn_major;
  g.colsum = p->colsum_partial;
  if (p->colsum_partial)
    HBA_REQUIRE(p->out_bf16 && !p->transpose_out && p->N % 4 == 0 && ((uintptr_t)p->colsum_partial & 15) == 0,
                "hba_gemm_bf16: colsum_partial needs a bf16 output, N %% 4 == 0 and a 16-byte aligned buffer");
  g.k_slices = 1, g.slice_stride = 0;
  g.tail_first = 0, g.tail_f = 1;
  const int kblocks_total = (p->K + BK - 1) / BK;
  int slices = p->k_slices > 1 ? p->k_slices : 1;
  if (slices > kblocks_total) slices = kblocks_total;
  ReduceArgs red = {};
  if (slices > 1) {
    HBA_REQUIRE(p->k_workspace && !p->transpose_out && !p->colsum_partial && p->N % 4 == 0,
                "hba_gemm_bf16: split-K (k_slices=%d) needs k_workspace, N %% 4 == 0 and no transposed / column-sum "
                "output", p->k_slices);
    HBA_REQUIRE(((uintptr_t)p->k_workspace & 15) == 0, "hba_gemm_bf16: k_workspace must be 16-byte aligned");
    // every slice must own at least one k-block
    const int kb_per = (kblocks_total + slices - 1) / slices;
    slices = (kblocks_total + kb_per - 1) / kb_per;
    g.k_slices = slices;
    g.slice_stride = (size_t)p->M * p->N;
    // the slices write plain fp32 partial sums (alpha applied); the epilogue proper runs in the reduction
    red.part = p->k_workspace, red.slice_stride = g.slice_stride, red.slices = slices;
    red.rows = p->M, red.cols = p->N, red.ld = p->N;
    red.bias = g.bias, red.residual = g.residual, red.ldr = g.ldr;
    red.act = g.act, red.aux = g.aux, red.ld_aux = g.ld_aux, red.aux_dtype = g.aux_dtype;
    red.pre_out = g.pre_out, red.ld_pre = g.ld_pre, red.pre_dtype = g.pre_dtype;
    red.out_f32 = g.out_f32, red.ld_f32 = g.ld_f32;
    red.out_bf16 = g.out_bf16, red.ld_bf16 = g.ld_bf16, red.out_lo_off = g.out_lo_off;
    g.bias = nullptr, g.residual = nullptr, g.act = HBA_ACT_NONE, g.aux = nullptr, g.pre_out = nullptr;
    g.out_bf16 = nullptr, g.out_lo_off = 0;
    g.out_f32 = p->k_workspace;
    g.ld_f32 = p->N;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool wide = p->N >= 256;
  if (g.k_slices > 1) {
    const int rc = wide ? launch_gemm<256, HBA_ACT_NONE>(p, g, s) : launch_gemm<128, HBA_ACT_NONE>(p, g, s);
    if (rc != HBA_OK) return rc;
    const size_t n4 = (size_t)p->M * (p->N / 4);
    int blocks = (int)((n4 + 255) / 256);
    if (blocks > 8 * num_sms()) blocks = 8 * num_sms();
    splitk_reduce_kernel<<<blocks, 256, 0, s>>>(red);
    return check_launch("splitk_reduce_kernel");
  }
  switch (p->act) {
#define HBA_GEMM_CASE(A) \
  case A:                \
    return wide ? launch_gemm<256, A>(p, g, s) : launch_gemm<128, A>(p, g, s);
    HBA_GEMM_CASE(HBA_ACT_NONE)
    HBA_GEMM_CASE(HBA_ACT_QUICKGELU)
    HBA_GEMM_CASE(HBA_ACT_GELU_ERF)
    HBA_GEMM_CASE(HBA_ACT_QUICKGELU_GRAD)
    HBA_GEMM_CASE(HBA_ACT_GELU_ERF_GRAD)
#undef HBA_GEMM_CASE
  }
  return HBA_ERR_ARG;  // (unreachable: act was checked above)
}
