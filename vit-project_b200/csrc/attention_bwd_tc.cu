// Softmax-attention backward on the tcgen05 tensor pipe (bf16 mode), head_dim 64, T <= 256.
// Reference semantics: autograd of F.multi_head_attention_forward -> SDPA (torch/nn/functional.py:6682),
// reached by the ViT-B/16 training step (Training/vit_training/baseline/train_vit_sgd.py:138-145).
//
// Persistent kernel, one CTA per SM, looping over (sequence, head) units.  The unit's Q, K, V and dO
// rows are fetched by TMA out of the packed [B*T, 3*H*64] QKV activation and the [B*T, H*64] output
// gradient, both addressed as [B, T, cols] so that rows past a sequence's end read as zero.  Keys are the TMEM lanes (one thread per key), queries the TMEM columns, so the two
// "transposed" products dV = P^T dO and dK = dS^T Q take their A operand straight from tensor memory:
//
//   per key tile t (128 keys) and query half h (<= 128 queries):
//     S^T  = K_t Q_h^T          UMMA 128 x N x 64, smem x smem          -> TMEM [0, 128)
//     dP^T = V_t dO_h^T         UMMA 128 x N x 64, smem x smem          -> TMEM [128, 256)
//     P^T  = 2^(S^T * scale - lse_i),  dS^T = P^T o (dP^T - D_i)        (8 warps: two column ranges)
//            written back as packed bf16 over S^T / dP^T, dS^T also to shared memory (MN-major A tile)
//     dV_t += P^T dO_h          UMMA 128 x 64 x N, A from TMEM, B = dO as loaded (MN-major)
//     dK_t += dS^T Q_h          UMMA 128 x 64 x N, A from TMEM, B = Q as loaded (MN-major)
//     dQ_h += dS K_t            UMMA 128 x 64 x 128, A = staged dS^T (MN-major), B = K as loaded
//
// lse_i (log2 domain, written by the forward kernel) and D_i = dO_i . O_i (computed here from the
// forward's bf16 output) are broadcast from shared memory.  The softmax scale 1/8 is applied to dQ and
// dK in the fp32 epilogue.
//
//   warp 0      TMA producer            warps 2..5   softmax / epilogue, first column range
//   warp 1      UMMA issuer, TMEM owner warps 6..9   softmax / epilogue, second column range
#include "common.cuh"

namespace hba {

namespace {

constexpr int kHd = 64;
constexpr int kRowBytes = 128;                 // 64 bf16
constexpr int kMaxRows = 256;                  // rows staged per operand
constexpr int kTileBytes = kMaxRows * kRowBytes;   // 32 KB per operand (Q, K, V, dO)
constexpr int kStageBytes = 2 * 128 * kRowBytes;   // dS^T tile: 2 blocks of (128 keys x 64 queries)
constexpr int kThreads = 320;
constexpr int kComputeThreads = 256;
constexpr int kBarBytes = 128;
constexpr int kSmemBytes = 4 * kTileBytes + kStageBytes + 2 * kMaxRows * 4 + kBarBytes + 1024;
constexpr int kTmemCols = 512;
constexpr int kColS = 0, kColDP = 128, kColDV = 256, kColDK = 320, kColDQ = 384;  // dQ_h at kColDQ + 64 h

__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_x8(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait_all() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}
__device__ __forceinline__ float dot_bf16x8(uint4 a, uint4 b) {
  const float2 a0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&a.x));
  const float2 a1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&a.y));
  const float2 a2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&a.z));
  const float2 a3 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&a.w));
  const float2 b0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&b.x));
  const float2 b1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&b.y));
  const float2 b2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&b.z));
  const float2 b3 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&b.w));
  return a0.x * b0.x + a0.y * b0.y + a1.x * b1.x + a1.y * b1.y + a2.x * b2.x + a2.y * b2.y +
         a3.x * b3.x + a3.y * b3.y;
}
// 32 fp32 accumulator columns of one row -> scaled bf16, 64 contiguous bytes
__device__ __forceinline__ void store_row32(const uint32_t* v, float scale, __nv_bfloat16* dst) {
  uint4* out = reinterpret_cast<uint4*>(dst);
#pragma unroll
  for (int j = 0; j < 4; ++j)
    out[j] = make_uint4(
        pack_bf16x2(__uint_as_float(v[8 * j]) * scale, __uint_as_float(v[8 * j + 1]) * scale),
        pack_bf16x2(__uint_as_float(v[8 * j + 2]) * scale, __uint_as_float(v[8 * j + 3]) * scale),
        pack_bf16x2(__uint_as_float(v[8 * j + 4]) * scale, __uint_as_float(v[8 * j + 5]) * scale),
        pack_bf16x2(__uint_as_float(v[8 * j + 6]) * scale, __uint_as_float(v[8 * j + 7]) * scale));
}
__device__ __forceinline__ void fence_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void compute_barrier() {
  asm volatile("bar.sync 1, %0;" ::"n"(kComputeThreads) : "memory");
}

struct AttnBwdArgs {
  int T, H, causal;
  int n_units;    // B * H
  int rows;       // rows staged per operand: T rounded up to 16
  int n_tiles;    // 128-row tiles (keys and queries): 1 or 2
  float scale_log2;
  const __nv_bfloat16* o;
  int64_t ld_o;
  const float* lse;   // [B, H, T], log2 domain (attention_tc_kernel)
  __nv_bfloat16* d_qkv;
  int64_t ld_dqkv;
};

// first column of the second warp group's range inside a half of n columns
__device__ __forceinline__ int split_col(int n) { return ((n >> 1) + 15) & ~15; }
// TMEM column (relative to the S^T / dP^T region) of the packed bf16 pairs of columns [c, c + 16)
__device__ __forceinline__ int packed_col(int c, int c1) { return c < c1 ? (c >> 1) : c1 + ((c - c1) >> 1); }

__global__ void __launch_bounds__(kThreads, 1)
    attention_bwd_tc_kernel(const __grid_constant__ CUtensorMap tma_qkv0,
                            const __grid_constant__ CUtensorMap tma_qkv1,
                            const __grid_constant__ CUtensorMap tma_do0,
                            const __grid_constant__ CUtensorMap tma_do1, const AttnBwdArgs g) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + kTileBytes;
  uint8_t* sV = sK + kTileBytes;
  uint8_t* sDO = sV + kTileBytes;
  uint8_t* sStage = sDO + kTileBytes;
  float* sL = reinterpret_cast<float*>(sStage + kStageBytes);
  float* sD = sL + kMaxRows;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sD + kMaxRows);
  uint64_t* in_full = bars;       // unit operands landed (TMA bytes)
  uint64_t* s_full = bars + 1;    // S^T and dP^T of the iteration complete
  uint64_t* p_full = bars + 2;    // P^T / dS^T written by the 8 compute warps
  uint64_t* acc_done = bars + 3;  // dV / dK / dQ UMMAs of the iteration complete
  uint64_t* in_empty = bars + 4;  // every UMMA of the unit has read its operands
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);
  const uint32_t smem_base = smem_u32(smem);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int d = g.H * kHd;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tma_qkv0);
    tma_prefetch_desc(&tma_qkv1);
    tma_prefetch_desc(&tma_do0);
    tma_prefetch_desc(&tma_do1);
    mbar_init(in_full, 1);
    mbar_init(s_full, 1);
    mbar_init(p_full, 8);
    mbar_init(acc_done, 1);
    mbar_init(in_empty, 1);
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int my_units = (g.n_units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int rows0 = g.rows < 128 ? g.rows : 128, rows1 = g.rows - rows0;

  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer
    const uint32_t bytes = (uint32_t)(4 * g.rows * kRowBytes);
    for (int n = 0; n < my_units; ++n) {
      const int u = blockIdx.x + n * gridDim.x;
      const int b = u / g.H, h = u % g.H;
      // every UMMA of the previous unit has read shared memory (and so have the compute warps, which
      // arrive on p_full after their last generic-proxy reads)
      if (n > 0) mbar_wait(in_empty, (uint32_t)((n - 1) & 1));
      if (elect_one()) {
        mbar_arrive_expect_tx(in_full, bytes);
        tma_load_3d(sQ, &tma_qkv0, in_full, h * kHd, 0, b);
        tma_load_3d(sK, &tma_qkv0, in_full, d + h * kHd, 0, b);
        tma_load_3d(sV, &tma_qkv0, in_full, 2 * d + h * kHd, 0, b);
        tma_load_3d(sDO, &tma_do0, in_full, h * kHd, 0, b);
        if (rows1 > 0) {
          tma_load_3d(sQ + 128 * kRowBytes, &tma_qkv1, in_full, h * kHd, 128, b);
          tma_load_3d(sK + 128 * kRowBytes, &tma_qkv1, in_full, d + h * kHd, 128, b);
          tma_load_3d(sV + 128 * kRowBytes, &tma_qkv1, in_full, 2 * d + h * kHd, 128, b);
          tma_load_3d(sDO + 128 * kRowBytes, &tma_do1, in_full, h * kHd, 128, b);
        }
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- UMMA issuer
    const uint32_t idesc_ts = make_idesc_bf16(128, kHd) | (1u << 16);              // B MN-major
    const uint32_t idesc_dq = make_idesc_bf16(128, kHd) | (1u << 15) | (1u << 16);  // A and B MN-major
    const uint64_t stage_lbo = (uint64_t)((128 * kRowBytes) >> 4) << 16;  // next 64-query block: 16 KB
    uint64_t stage_desc = make_smem_desc_sw128(smem_u32(sStage));
    stage_desc = (stage_desc & ~((uint64_t)0x3FFF << 16)) | stage_lbo;
    int git = 0;
    for (int n = 0; n < my_units; ++n) {
      mbar_wait(in_full, (uint32_t)(n & 1));
      tc_fence_after();
      for (int t = 0; t < g.n_tiles; ++t) {
        const int nk = t == 0 ? rows0 : rows1;  // keys of the tile (multiple of 16)
        for (int hh = 0; hh < g.n_tiles; ++hh, ++git) {
          const int nq = hh == 0 ? rows0 : rows1;  // queries of the half
          const int c1 = split_col(nq);
          // P^T / dS^T of the previous iteration have been consumed
          if (git > 0) {
            mbar_wait(acc_done, (uint32_t)((git - 1) & 1));
            tc_fence_after();
          }
          if (elect_one()) {
            const uint32_t idesc_s = make_idesc_bf16(128, nq);
            const uint64_t k_desc = make_smem_desc_sw128(smem_u32(sK + t * 128 * kRowBytes));
            const uint64_t v_desc = make_smem_desc_sw128(smem_u32(sV + t * 128 * kRowBytes));
            const uint64_t q_desc = make_smem_desc_sw128(smem_u32(sQ + hh * 128 * kRowBytes));
            const uint64_t do_desc = make_smem_desc_sw128(smem_u32(sDO + hh * 128 * kRowBytes));
#pragma unroll
            for (int k = 0; k < kHd / 16; ++k)
              umma_bf16(tmem_base + kColS, k_desc + 2 * k, q_desc + 2 * k, idesc_s, k > 0 ? 1u : 0u);
#pragma unroll
            for (int k = 0; k < kHd / 16; ++k)
              umma_bf16(tmem_base + kColDP, v_desc + 2 * k, do_desc + 2 * k, idesc_s, k > 0 ? 1u : 0u);
            umma_commit(s_full);
          }
          __syncwarp();
          mbar_wait(p_full, (uint32_t)(git & 1));
          tc_fence_after();
          if (elect_one()) {
            const uint64_t do_desc = make_smem_desc_sw128(smem_u32(sDO + hh * 128 * kRowBytes));
            const uint64_t q_desc = make_smem_desc_sw128(smem_u32(sQ + hh * 128 * kRowBytes));
            const uint64_t k_desc = make_smem_desc_sw128(smem_u32(sK + t * 128 * kRowBytes));
            for (int kk = 0; kk < nq / 16; ++kk) {
              const uint32_t pc = (uint32_t)packed_col(16 * kk, c1);
              umma_ts(tmem_base + kColDV, tmem_base + kColS + pc, do_desc + (uint64_t)(kk * 128),
                      idesc_ts, (hh > 0 || kk > 0) ? 1u : 0u);
            }
            for (int kk = 0; kk < nq / 16; ++kk) {
              const uint32_t pc = (uint32_t)packed_col(16 * kk, c1);
              umma_ts(tmem_base + kColDK, tmem_base + kColDP + pc, q_desc + (uint64_t)(kk * 128),
                      idesc_ts, (hh > 0 || kk > 0) ? 1u : 0u);
            }
            for (int kk = 0; kk < nk / 16; ++kk)
              umma_bf16(tmem_base + kColDQ + 64 * hh, stage_desc + (uint64_t)(kk * 128),
                        k_desc + (uint64_t)(kk * 128), idesc_dq, (t > 0 || kk > 0) ? 1u : 0u);
            umma_commit(acc_done);
            if (t == g.n_tiles - 1 && hh == g.n_tiles - 1) umma_commit(in_empty);
          }
          __syncwarp();
        }
      }
    }
    // the last commit must have completed before TMEM is released
    if (git > 0) mbar_wait(acc_done, (uint32_t)((git - 1) & 1));
  } else {
    // ---------------------------------------------------------------- softmax + epilogue
    const int wg = (warp - 2) >> 2;    // column range served by this warp group
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;       // key row inside the tile = TMEM lane
    const int ct = (warp - 2) * 32 + lane;  // compute-thread index: query row whose D_i it prepares
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t stage_base = smem_u32(sStage);
    const uint32_t sL_base = smem_u32(sL), sD_base = smem_u32(sD), sDO_base = smem_u32(sDO);
    int git = 0;
    for (int n = 0; n < my_units; ++n) {
      const int u = blockIdx.x + n * gridDim.x;
      const int b = u / g.H, h = u % g.H;
      // ---- D_i = dO_i . O_i, lse_i -> shared memory
      uint4 ov[8];
      float my_lse = 0.f;
      if (ct < g.T) {
        const uint4* orow = reinterpret_cast<const uint4*>(g.o + ((int64_t)b * g.T + ct) * g.ld_o + h * kHd);
#pragma unroll
        for (int c = 0; c < 8; ++c) ov[c] = __ldg(orow + c);
        my_lse = __ldg(g.lse + ((int64_t)b * g.H + h) * g.T + ct);
      }
      mbar_wait(in_full, (uint32_t)(n & 1));
      float my_d = 0.f;
      if (ct < g.T) {
#pragma unroll
        for (int c = 0; c < 8; ++c)
          my_d += dot_bf16x8(ov[c], lds128(sDO_base + ct * kRowBytes + ((c ^ (ct & 7)) << 4)));
      }
      sL[ct] = my_lse;
      sD[ct] = my_d;
      compute_barrier();
      for (int t = 0; t < g.n_tiles; ++t) {
        const int kj = t * 128 + r;  // key index inside the sequence
        const bool key_ok = kj < g.T;
        for (int hh = 0; hh < g.n_tiles; ++hh, ++git) {
          const int nq = hh == 0 ? rows0 : rows1;
          const int c1 = split_col(nq);
          const int c_lo = wg == 0 ? 0 : c1, c_hi = wg == 0 ? c1 : nq;
          mbar_wait(s_full, (uint32_t)(git & 1));
          tc_fence_after();
          auto process = [&](const uint32_t* sv, const uint32_t* dpv, int c) {
            const int qi0 = hh * 128 + c;  // first query of the chunk
            float lse[16], dd[16];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 a = lds128(sL_base + 4 * (qi0 + 4 * j));
              const uint4 e = lds128(sD_base + 4 * (qi0 + 4 * j));
              lse[4 * j] = __uint_as_float(a.x), lse[4 * j + 1] = __uint_as_float(a.y);
              lse[4 * j + 2] = __uint_as_float(a.z), lse[4 * j + 3] = __uint_as_float(a.w);
              dd[4 * j] = __uint_as_float(e.x), dd[4 * j + 1] = __uint_as_float(e.y);
              dd[4 * j + 2] = __uint_as_float(e.z), dd[4 * j + 3] = __uint_as_float(e.w);
            }
            float p[16], ds[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              p[j] = ex2f(fmaf(__uint_as_float(sv[j]), g.scale_log2, -lse[j]));
              ds[j] = p[j] * (__uint_as_float(dpv[j]) - dd[j]);
              const bool ok = key_ok && (qi0 + j < g.T) && (!g.causal || kj <= qi0 + j);
              p[j] = ok ? p[j] : 0.f;
              ds[j] = ok ? ds[j] : 0.f;
            }
            uint32_t pk[8], dk[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              pk[j] = pack_bf16x2(p[2 * j], p[2 * j + 1]);
              dk[j] = pack_bf16x2(ds[2 * j], ds[2 * j + 1]);
            }
            const uint32_t pc = (uint32_t)packed_col(c, c1);
            tmem_st_x8(lane_addr + kColS + pc, pk);
            tmem_st_x8(lane_addr + kColDP + pc, dk);
            // dS^T (key r, queries c..c+15) -> MN-major tile: block c / 64, row r, 16-byte chunks
            const uint32_t row_addr = stage_base + (uint32_t)(c >> 6) * (128 * kRowBytes) + r * kRowBytes;
            const int ch = (c & 63) >> 3;
            sts128(row_addr + ((ch ^ (r & 7)) << 4), dk[0], dk[1], dk[2], dk[3]);
            sts128(row_addr + (((ch + 1) ^ (r & 7)) << 4), dk[4], dk[5], dk[6], dk[7]);
          };
          {
            uint32_t sa[16], da[16], sb[16], db[16];
            if (c_lo < c_hi) {
              tmem_ld_x16(lane_addr + kColS + c_lo, sa);
              tmem_ld_x16(lane_addr + kColDP + c_lo, da);
            }
#pragma unroll 1
            for (int c = c_lo; c < c_hi; c += 32) {
              tmem_ld_wait();
              if (c + 16 < c_hi) {
                tmem_ld_x16(lane_addr + kColS + c + 16, sb);
                tmem_ld_x16(lane_addr + kColDP + c + 16, db);
              }
              process(sa, da, c);
              if (c + 16 < c_hi) {
                tmem_ld_wait();
                if (c + 32 < c_hi) {
                  tmem_ld_x16(lane_addr + kColS + c + 32, sa);
                  tmem_ld_x16(lane_addr + kColDP + c + 32, da);
                }
                process(sb, db, c + 16);
              }
            }
          }
          tmem_st_wait_all();
          fence_async_smem();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(p_full);
          // ---- epilogues: every accumulator's 64 columns are split between the two warp groups
          mbar_wait(acc_done, (uint32_t)(git & 1));
          tc_fence_after();
          if (hh == g.n_tiles - 1) {  // dV_t, dK_t complete: rows = keys of the tile
            // (tcgen05.ld is warp-collective: every lane loads, only valid rows store)
            __nv_bfloat16* row = g.d_qkv + ((int64_t)b * g.T + (key_ok ? kj : 0)) * g.ld_dqkv + h * kHd + 32 * wg;
            uint32_t v[32];
            tmem_ld_32x32b_x32(lane_addr + kColDK + 32 * wg, v);
            tmem_ld_wait();
            if (key_ok) store_row32(v, 0.125f, row + d);
            tmem_ld_32x32b_x32(lane_addr + kColDV + 32 * wg, v);
            tmem_ld_wait();
            if (key_ok) store_row32(v, 1.0f, row + 2 * d);
          }
          if (t == g.n_tiles - 1) {  // dQ_h complete: rows = queries of the half
            const int qi = hh * 128 + r;
            uint32_t v[32];
            tmem_ld_32x32b_x32(lane_addr + kColDQ + 64 * hh + 32 * wg, v);
            tmem_ld_wait();
            if (qi < g.T)
              store_row32(v, 0.125f, g.d_qkv + ((int64_t)b * g.T + qi) * g.ld_dqkv + h * kHd + 32 * wg);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

}  // namespace

// host launcher, called from hba_attention_bwd_lse (attention.cu)
int attention_bwd_tc_launch(const __nv_bfloat16* qkv, int64_t ld_qkv, int B, int T, int H, int causal,
                            const __nv_bfloat16* o, int64_t ld_o, const __nv_bfloat16* d_out, int64_t ld_do,
                            const float* lse, __nv_bfloat16* d_qkv, int64_t ld_dqkv, cudaStream_t stream) {
  static SmemAttr attr;
  HBA_CHECK(ensure_dyn_smem(attention_bwd_tc_kernel, kSmemBytes, attr, "attention_bwd_tc_kernel"));
  if (T > kMaxRows) {
    set_error("attention_bwd_tc: T=%d exceeds %d", T, kMaxRows);
    return HBA_ERR_ARG;
  }
  AttnBwdArgs g;
  g.T = T, g.H = H, g.causal = causal;
  g.n_units = B * H;
  g.rows = (T + 15) / 16 * 16;
  g.n_tiles = g.rows > 128 ? 2 : 1;
  g.scale_log2 = 1.4426950408889634f * 0.125f;
  g.o = o, g.ld_o = ld_o, g.lse = lse, g.d_qkv = d_qkv, g.ld_dqkv = ld_dqkv;
  const uint32_t rows0 = g.rows < 128 ? g.rows : 128;
  const uint32_t rows1 = g.rows > 128 ? g.rows - 128 : 16;  // (unused map when there is one tile)
  // [B, T, cols] maps: rows >= T of a sequence (the boxes are T rounded up to 16) read as zero, not as the
  // next sequence's first rows, whose non-finite values would survive the P / dS = 0 masking
  CUtensorMap q0, q1, d0, d1;
  HBA_CHECK(make_tma_3d_bf16(&q0, qkv, B, T, (uint64_t)3 * H * kHd, ld_qkv, rows0, 64));
  HBA_CHECK(make_tma_3d_bf16(&q1, qkv, B, T, (uint64_t)3 * H * kHd, ld_qkv, rows1, 64));
  HBA_CHECK(make_tma_3d_bf16(&d0, d_out, B, T, (uint64_t)H * kHd, ld_do, rows0, 64));
  HBA_CHECK(make_tma_3d_bf16(&d1, d_out, B, T, (uint64_t)H * kHd, ld_do, rows1, 64));
  int ctas = num_sms();
  if (g.n_units < ctas) ctas = g.n_units;
  attention_bwd_tc_kernel<<<ctas, kThreads, kSmemBytes, stream>>>(q0, q1, d0, d1, g);
  return check_launch("attention_bwd_tc_kernel");
}

}  // namespace hba
