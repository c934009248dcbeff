// Fused softmax attention on the tcgen05 tensor pipe (bf16 mode), head_dim 64, T <= 257.
// Reference semantics: F.multi_head_attention_forward -> SDPA (torch/nn/functional.py:6682).
//
// Persistent kernel, one CTA per SM, looping over (sequence, head) units; a unit is one or two
// 128-row query tiles ("items").  Everything a unit needs (its Q tiles and all K / V rows) is fetched
// by TMA straight out of the packed [B*T, 3*H*64] bf16 QKV activation (addressed as [B, T, 3*H*64], so
// that rows past a sequence's end read as zero) into one of two shared-memory buffers, so the loads of unit u+1 overlap the math of unit u.
//
//   S = Q K^T   UMMA 128 x NK x 64 (A, B from smem, SWIZZLE_128B K-major), fp32 in TMEM
//   softmax     one thread per query row: tcgen05.ld S, max, exp2 on the SFU, P packed to bf16 and
//               written BACK INTO TMEM over S (tcgen05.st) - P never touches shared memory
//   O = P V     UMMA 128 x 64 x NK with A = P from TMEM and B = V as loaded (MN-major descriptor)
//
// TMEM is split into two 256-column regions; item i uses region i & 1 and softmax warp-group i & 1, so
// the softmax of one item runs while the tensor pipe produces S / O of the other one.
// T = 257 = 2*128 + 1 (CLIP ViT-L/14): keys 0..255 go through the tensor cores; key 256 is added by
// the row's own thread in fp32, and query row 256 (T mod 128 <= 8 left-over
// rows) is computed by two CUDA-core warps from the same shared-memory K / V tiles.
//
//   warp 0      TMA producer                   warps 2..5   softmax + epilogue, even items (region 0)
//   warp 1      UMMA issuer, TMEM owner        warps 6..9   softmax + epilogue, odd items  (region 1)
//                                              warps 10..11 left-over query rows (CUDA cores)
#include "common.cuh"

namespace hba {

constexpr int kTcHd = 64;
constexpr int kTcRowBytes = 128;               // 64 bf16
constexpr int kTcQBytes = 128 * kTcRowBytes;   // 16 KB per Q tile
constexpr int kTcMaxRows = 272;                // K / V rows staged per unit
constexpr int kTcKVBytes = kTcMaxRows * kTcRowBytes;         // 34 KB
constexpr int kTcBufBytes = 2 * kTcQBytes + 2 * kTcKVBytes;  // 100 KB per unit buffer
constexpr int kTcThreads = 384;
constexpr int kTcBarBytes = 256;
constexpr int kTcLeftFloats = 2 * (kTcMaxRows + kTcHd);
constexpr int kTcSmemBytes = 2 * kTcBufBytes + kTcBarBytes + kTcLeftFloats * 4 + 1024;
constexpr int kTcTmemCols = 512;
constexpr int kTcRegionCols = 256;
constexpr int kTcOCol = 128;  // O accumulator columns [128, 192) of the region (P packs into [0, 128))
constexpr int kTcMaxExtra = 1;   // T = 257: one key beyond the 256 tensor-core keys

__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 8 columns: thread t writes its 8 registers into lane (base_lane + t)
__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, "
      "%13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
      "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]: the A operand (P, bf16 pairs packed in 32-bit columns) is read
// from tensor memory
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b,
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
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// instruction descriptor: bf16 A (K-major) x bf16 B (K-major or MN-major), fp32 accumulate
__device__ __forceinline__ uint32_t idesc_bf16(int M, int N, bool b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (b_mn_major ? (1u << 16) : 0u) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// byte offset of element (row, col) inside a [rows x 64] bf16 SWIZZLE_128B tile
__device__ __forceinline__ uint32_t sw128_off(int row, int col) {
  return (uint32_t)row * 128u + ((((uint32_t)col >> 3) ^ ((uint32_t)row & 7u)) << 4) +
         (((uint32_t)col & 7u) << 1);
}
__device__ __forceinline__ uint4 lds_u4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "r"(addr));
  return v;
}
__device__ __forceinline__ float4 lds128f(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ float2 bf2_to_f2(uint32_t u) {
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u));
}

struct AttnTcArgs {
  int T, H, causal;
  int n_units;     // B * H
  int n_tiles;     // 128-row query tiles on the tensor cores (1 or 2)
  int n_left;      // left-over query rows (CUDA cores), rows [128*n_tiles, T)
  int NK;          // keys on the tensor cores (multiple of 16, <= 256)
  int n_extra;     // keys [NK, T) added in fp32 by the row threads (T > 256 only)
  int kv_rows;     // K / V rows staged per unit (multiple of 16, >= T)
  __nv_bfloat16* out;
  int64_t ld_out;
  float* out_f32;
  int64_t ld_of;
  float scale_log2;  // log2(e) / sqrt(64)
  const __nv_bfloat16* qkv;
  int64_t ld_qkv;
  float* lse;        // optional [B, H, T]: log2-domain log-sum-exp per row (P = 2^(s*scale - lse)), for the backward
};

__global__ void __launch_bounds__(kTcThreads, 1)
    attention_tc_kernel(const __grid_constant__ CUtensorMap tma128,
                        const __grid_constant__ CUtensorMap tma16, const AttnTcArgs g) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  // buffer b: Q tile 0, Q tile 1, K, V
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * kTcBufBytes);
  uint64_t* kv_full = bars;        // [2] unit buffer landed (TMA bytes)
  uint64_t* kv_empty = bars + 2;   // [2] every reader of the buffer is done
  uint64_t* s_full = bars + 4;     // [2] S of the region's item complete
  uint64_t* p_full = bars + 6;     // [2] P written to TMEM by the 4 softmax warps
  uint64_t* o_full = bars + 8;     // [2] O complete
  uint64_t* r_free = bars + 10;    // [2] O read out: the region may take the next S
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t left_base = smem_base + 2 * kTcBufBytes + kTcBarBytes;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // warp-uniform role dispatch
  const int lane = threadIdx.x & 31;
  const int d = g.H * kTcHd;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tma128);
    tma_prefetch_desc(&tma16);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1 + 4 * g.n_tiles + 2);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 4);
      mbar_init(&o_full[i], 1);
      mbar_init(&r_free[i], 4);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, kTcTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // units of this CTA: u = blockIdx.x + n * gridDim.x, n = 0 .. my_units-1
  const int my_units = (g.n_units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int my_items = my_units * g.n_tiles;

  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer
    const int full = g.kv_rows / 128, tail = (g.kv_rows % 128) / 16;
    const uint32_t bytes = (uint32_t)(g.n_tiles * kTcQBytes + 2 * g.kv_rows * kTcRowBytes);
    for (int n = 0; n < my_units; ++n) {
      const int u = blockIdx.x + n * gridDim.x;
      const int b = u / g.H, h = u % g.H;
      const int buf = n & 1;
      mbar_wait(&kv_empty[buf], ((n >> 1) & 1) ^ 1);
      if (elect_one()) {
        uint8_t* sQ = smem + buf * kTcBufBytes;
        uint8_t* sK = sQ + 2 * kTcQBytes;
        uint8_t* sV = sK + kTcKVBytes;
        mbar_arrive_expect_tx(&kv_full[buf], bytes);
        for (int t = 0; t < g.n_tiles; ++t)
          tma_load_3d(sQ + t * kTcQBytes, &tma128, &kv_full[buf], h * kTcHd, t * 128, b);
        for (int i = 0; i < full; ++i) {
          tma_load_3d(sK + i * kTcQBytes, &tma128, &kv_full[buf], d + h * kTcHd, i * 128, b);
          tma_load_3d(sV + i * kTcQBytes, &tma128, &kv_full[buf], 2 * d + h * kTcHd, i * 128, b);
        }
        for (int i = 0; i < tail; ++i) {
          const int r = full * 128 + i * 16;
          tma_load_3d(sK + r * kTcRowBytes, &tma16, &kv_full[buf], d + h * kTcHd, r, b);
          tma_load_3d(sV + r * kTcRowBytes, &tma16, &kv_full[buf], 2 * d + h * kTcHd, r, b);
        }
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- UMMA issuer
    const uint32_t idesc_s = idesc_bf16(128, g.NK, false);
    const uint32_t idesc_o = idesc_bf16(128, kTcHd, true);
    auto issue_pv = [&](int j) {  // O(j) = P(j) V once the softmax group has written P(j)
      const int n = j / g.n_tiles, tile = j - n * g.n_tiles;
      const int region = j & 1, buf = n & 1;
      mbar_wait(&p_full[region], (j >> 1) & 1);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t tP = tmem_base + region * kTcRegionCols, tO = tP + kTcOCol;
        const uint64_t v_desc =
            make_smem_desc_sw128(smem_base + buf * kTcBufBytes + 2 * kTcQBytes + kTcKVBytes);
        for (int kk = 0; kk < g.NK / 16; ++kk)
          umma_bf16_ts(tO, tP + kk * 8, v_desc + (uint64_t)(kk * 16 * kTcRowBytes >> 4), idesc_o,
                       kk > 0 ? 1u : 0u);
        umma_commit(&o_full[region]);
        if (tile == g.n_tiles - 1) umma_commit(&kv_empty[buf]);  // every UMMA of the unit has read smem
      }
      __syncwarp();
    };
    for (int i = 0; i < my_items; ++i) {
      const int n = i / g.n_tiles, tile = i - n * g.n_tiles;
      const int region = i & 1, buf = n & 1;
      if (tile == 0) mbar_wait(&kv_full[buf], (n >> 1) & 1);
      // Stagger the two softmax groups by half a period: the very first odd item starts only when
      // the even group has finished its exp pass, so that from then on one group runs its SFU-bound
      // exp pass while the other is in its max pass / epilogue / waiting for the tensor pipe
      // (in lock-step both groups fought for the SFU and then left it idle together: 40 % busy).
      if (i == 1) mbar_wait(&p_full[0], 0);
      mbar_wait(&r_free[region], ((i >> 1) & 1) ^ 1);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t q_addr = smem_base + buf * kTcBufBytes + tile * kTcQBytes;
        const uint64_t q_desc = make_smem_desc_sw128(q_addr);
        const uint64_t k_desc = make_smem_desc_sw128(smem_base + buf * kTcBufBytes + 2 * kTcQBytes);
        const uint32_t tS = tmem_base + region * kTcRegionCols;
#pragma unroll
        for (int k = 0; k < kTcHd / 16; ++k)
          umma_bf16(tS, q_desc + 2 * k, k_desc + 2 * k, idesc_s, k > 0 ? 1u : 0u);
        umma_commit(&s_full[region]);
      }
      __syncwarp();
      if (i >= 1) issue_pv(i - 1);
    }
    if (my_items > 0) issue_pv(my_items - 1);
  } else if (warp < 10) {
    // ---------------------------------------------------------------- softmax + epilogue
    const int grp = (warp - 2) >> 2;   // region / item parity served by this warp group
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;       // query row inside the tile = TMEM lane
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + grp * kTcRegionCols;
    for (int i = grp; i < my_items; i += 2) {
      const int n = i / g.n_tiles, tile = i - n * g.n_tiles;
      const int buf = n & 1, use = i >> 1;
      const int u = blockIdx.x + n * gridDim.x;
      const int b = u / g.H, h = u % g.H;
      const int qi = tile * 128 + r;  // query index inside the sequence
      const int last_key = g.causal ? min(qi, g.T - 1) : g.T - 1;
      const uint32_t sQ = smem_base + buf * kTcBufBytes + tile * kTcQBytes;
      const uint32_t sK = smem_base + buf * kTcBufBytes + 2 * kTcQBytes;
      const uint32_t sV = sK + kTcKVBytes;
      // key NK (= 256, T = 257 only): s = q . k in fp32 from the staged tiles
      float s_extra = 0.f;
      float mx = -INFINITY;
      const bool extra_valid = g.n_extra > 0 && g.NK <= last_key;
      if (g.n_extra > 0) {
        mbar_wait(&kv_full[buf], (n >> 1) & 1);
        const int kr = g.NK;
#pragma unroll 2
        for (int c = 0; c < 8; ++c) {
          const uint4 qv = lds_u4(sQ + r * kTcRowBytes + ((c ^ (r & 7)) << 4));
          const uint4 kv = lds_u4(sK + kr * kTcRowBytes + ((c ^ (kr & 7)) << 4));
          const float2 q0 = bf2_to_f2(qv.x), q1 = bf2_to_f2(qv.y), q2 = bf2_to_f2(qv.z), q3 = bf2_to_f2(qv.w);
          const float2 k0 = bf2_to_f2(kv.x), k1 = bf2_to_f2(kv.y), k2 = bf2_to_f2(kv.z), k3 = bf2_to_f2(kv.w);
          s_extra += q0.x * k0.x + q0.y * k0.y + q1.x * k1.x + q1.y * k1.y + q2.x * k2.x + q2.y * k2.y +
                     q3.x * k3.x + q3.y * k3.y;
        }
        if (extra_valid) mx = s_extra;
      }
      const int nvalid = min(last_key + 1, g.NK);  // tensor-core keys this row attends to
      // tcgen05.ld / .st are warp-collective: loop bounds and branches below use warp-uniform counts
      const int nv_min = __reduce_min_sync(0xffffffffu, nvalid);
      const int nv_max = __reduce_max_sync(0xffffffffu, nvalid);
      mbar_wait(&s_full[grp], use & 1);
      tc_fence_after();
      // Both passes read S in 32-column chunks, double buffered: the tcgen05.ld of chunk k+1 is issued
      // (unconditionally, address clamped to the last chunk) before chunk k is processed, so a TMEM
      // round trip overlaps the math.  Four independent partial maxima / sums keep the dependent
      // FMNMX / FADD chains short.  Columns in [NK, roundup32(NK)) hold stale data: masked.
      const int c_last = ((nv_max + 31) & ~31) - 32;  // first column of the last chunk (>= 0)
      float m4[4] = {mx, -INFINITY, -INFINITY, -INFINITY};
      auto max32 = [&](const uint32_t* v, int c) {
        if (c + 32 <= nv_min) {
#pragma unroll
          for (int j = 0; j < 32; ++j) m4[j & 3] = fmaxf(m4[j & 3], __uint_as_float(v[j]));
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            m4[j & 3] = fmaxf(m4[j & 3], (c + j < nvalid) ? __uint_as_float(v[j]) : -INFINITY);
        }
      };
      {
        uint32_t va[32], vb[32];
        tmem_ld_32x32b_x32(lane_addr, va);
#pragma unroll 1
        for (int c = 0; c <= c_last; c += 64) {
          tmem_ld_wait();
          tmem_ld_32x32b_x32(lane_addr + min(c + 32, c_last), vb);
          max32(va, c);
          tmem_ld_wait();
          tmem_ld_32x32b_x32(lane_addr + min(c + 64, c_last), va);
          if (c + 32 <= c_last) max32(vb, c + 32);
        }
      }
      mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
      const float mxs = mx * g.scale_log2;
      // pass 2: p = 2^(s * scale - max * scale), packed to bf16 over the S columns already consumed
      float s4[4] = {0.f, 0.f, 0.f, 0.f};
      auto exp32 = [&](const uint32_t* v, int c) {
        uint32_t pk[16];
        float p[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) p[j] = ex2_approx(fmaf(__uint_as_float(v[j]), g.scale_log2, -mxs));
        if (c + 32 > nv_min) {
#pragma unroll
          for (int j = 0; j < 32; ++j) p[j] = (c + j < nvalid) ? p[j] : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 32; ++j) s4[j & 3] += p[j];
#pragma unroll
        for (int j = 0; j < 16; ++j) pk[j] = pack_bf16x2(p[2 * j], p[2 * j + 1]);
        tmem_st_32x32b_x16(lane_addr + (c >> 1), pk);
      };
      {
        uint32_t va[32], vb[32];
        tmem_ld_wait();  // (the clamped prefetch left over from pass 1)
        tmem_ld_32x32b_x32(lane_addr, va);
#pragma unroll 1
        for (int c = 0; c <= c_last; c += 64) {
          tmem_ld_wait();
          tmem_ld_32x32b_x32(lane_addr + min(c + 32, c_last), vb);
          exp32(va, c);
          tmem_ld_wait();
          // (chunk c + 64 is past every P column written so far: P(c + 32) ends at column c/2 + 32)
          tmem_ld_32x32b_x32(lane_addr + min(c + 64, c_last), va);
          if (c + 32 <= c_last) exp32(vb, c + 32);
        }
        tmem_ld_wait();
        // keys no row of this warp attends to (causal): P = 0
        uint32_t zero[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) zero[j] = 0u;
#pragma unroll 1
        for (int c = c_last + 32; c < g.NK; c += 32) tmem_st_32x32b_x16(lane_addr + (c >> 1), zero);
      }
      float sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[grp]);
      const float p_extra = extra_valid ? ex2_approx(fmaf(s_extra, g.scale_log2, -mxs)) : 0.f;
      sum += p_extra;
      if (g.lse && qi < g.T) g.lse[((int64_t)b * g.H + h) * g.T + qi] = mxs + __log2f(sum);
      // ---- O epilogue ----
      mbar_wait(&o_full[grp], use & 1);
      tc_fence_after();
      const float inv = __fdividef(1.0f, sum);
      const int64_t grow = (int64_t)b * g.T + qi;
      uint32_t o_all[64];
      tmem_ld_32x32b_x32(lane_addr + kTcOCol, o_all);
      tmem_ld_32x32b_x32(lane_addr + kTcOCol + 32, o_all + 32);
      tmem_ld_wait();
      // O is in registers: hand the TMEM region back before the (slower) store phase
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&r_free[grp]);
      float f[64];
#pragma unroll
      for (int j = 0; j < 64; ++j) f[j] = __uint_as_float(o_all[j]);
      if (g.n_extra > 0) {
        const int vr = g.NK;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const uint4 vv = lds_u4(sV + vr * kTcRowBytes + ((c ^ (vr & 7)) << 4));
          const float2 v0 = bf2_to_f2(vv.x), v1 = bf2_to_f2(vv.y), v2 = bf2_to_f2(vv.z), v3 = bf2_to_f2(vv.w);
          f[8 * c] += p_extra * v0.x, f[8 * c + 1] += p_extra * v0.y;
          f[8 * c + 2] += p_extra * v1.x, f[8 * c + 3] += p_extra * v1.y;
          f[8 * c + 4] += p_extra * v2.x, f[8 * c + 5] += p_extra * v2.y;
          f[8 * c + 6] += p_extra * v3.x, f[8 * c + 7] += p_extra * v3.y;
        }
      }
#pragma unroll
      for (int j = 0; j < 64; ++j) f[j] *= inv;
      if (g.out_f32 && qi < g.T) {  // fp32 copy (kept for the backward pass / trunk cache): row per thread
        float* dst = g.out_f32 + grow * g.ld_of + h * kTcHd;
#pragma unroll
        for (int j = 0; j < 64; j += 4)
          *reinterpret_cast<float4*>(dst + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
      }
      if (g.out) {
        // bf16 output: the warp's 32 rows are transposed through the (now dead) Q tile of this item so
        // that every store instruction writes 4 rows x 128 contiguous bytes instead of 32 rows x 16
#pragma unroll
        for (int c = 0; c < 8; ++c)
          asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(sQ + r * kTcRowBytes + ((c ^ (r & 7)) << 4)),
                       "r"(pack_bf16x2(f[8 * c], f[8 * c + 1])), "r"(pack_bf16x2(f[8 * c + 2], f[8 * c + 3])),
                       "r"(pack_bf16x2(f[8 * c + 4], f[8 * c + 5])), "r"(pack_bf16x2(f[8 * c + 6], f[8 * c + 7]))
                       : "memory");
        __syncwarp();
        const int cq = lane & 7, rsub = lane >> 3;
        uint4 ov[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int rl = q * 32 + 4 * k + rsub;
          ov[k] = lds_u4(sQ + rl * kTcRowBytes + ((cq ^ (rl & 7)) << 4));
        }
        __nv_bfloat16* obase = g.out + ((int64_t)b * g.T + tile * 128 + q * 32 + rsub) * g.ld_out + h * kTcHd + 8 * cq;
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (tile * 128 + q * 32 + 4 * k + rsub < g.T)
            *reinterpret_cast<uint4*>(obase + (int64_t)(4 * k) * g.ld_out) = ov[k];
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&kv_empty[buf]);
    }
  } else {
    // ---------------------------------------------------------------- left-over query rows (CUDA cores)
    const int w = warp - 10;
    const uint32_t pbuf = left_base + w * kTcMaxRows * 4;
    const uint32_t qbuf = left_base + 2 * kTcMaxRows * 4 + w * kTcHd * 4;
    for (int n = 0; n < my_units; ++n) {
      const int buf = n & 1;
      // always wait (also with no left-over rows): one kv_empty arrival per warp and per unit phase
      mbar_wait(&kv_full[buf], (n >> 1) & 1);
      if (g.n_left > 0) {
        const int u = blockIdx.x + n * gridDim.x;
        const int b = u / g.H, h = u % g.H;
        const uint32_t sK = smem_base + buf * kTcBufBytes + 2 * kTcQBytes;
        const uint32_t sV = sK + kTcKVBytes;
        for (int lr = w; lr < g.n_left; lr += 2) {
          const int qi = g.n_tiles * 128 + lr;
          const int last_key = g.causal ? min(qi, g.T - 1) : g.T - 1;
          // the query row is one of the staged K-tile rows' neighbours: read it from global (64 bf16)
          const __nv_bfloat16* qrow = g.qkv + ((int64_t)b * g.T + qi) * g.ld_qkv + h * kTcHd;
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(qbuf + 4 * lane), "f"(__bfloat162float(qrow[lane])) : "memory");
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(qbuf + 4 * (lane + 32)), "f"(__bfloat162float(qrow[lane + 32])) : "memory");
          __syncwarp();
          float s[(kTcMaxRows + 31) / 32];
          float mx = -INFINITY;
#pragma unroll
          for (int jj = 0; jj < (kTcMaxRows + 31) / 32; ++jj) {
            const int j = lane + 32 * jj;
            s[jj] = -INFINITY;
            if (j <= last_key) {
              float dot = 0.f;
#pragma unroll 2
              for (int c = 0; c < 8; ++c) {
                const uint4 kv = lds_u4(sK + j * kTcRowBytes + ((c ^ (j & 7)) << 4));
                const float4 qa = lds128f(qbuf + 32 * c), qb = lds128f(qbuf + 32 * c + 16);
                const float2 k0 = bf2_to_f2(kv.x), k1 = bf2_to_f2(kv.y), k2 = bf2_to_f2(kv.z), k3 = bf2_to_f2(kv.w);
                dot += qa.x * k0.x + qa.y * k0.y + qa.z * k1.x + qa.w * k1.y + qb.x * k2.x + qb.y * k2.y +
                       qb.z * k3.x + qb.w * k3.y;
              }
              s[jj] = dot;
              mx = fmaxf(mx, dot);
            }
          }
          mx = warp_max(mx);
          const float mxs = mx * g.scale_log2;
          float sum = 0.f;
#pragma unroll
          for (int jj = 0; jj < (kTcMaxRows + 31) / 32; ++jj) {
            const int j = lane + 32 * jj;
            const float p = (j <= last_key) ? ex2_approx(fmaf(s[jj], g.scale_log2, -mxs)) : 0.f;
            sum += p;
            if (j < kTcMaxRows) asm volatile("st.shared.f32 [%0], %1;" ::"r"(pbuf + 4 * j), "f"(p) : "memory");
          }
          sum = warp_sum(sum);
          if (g.lse && lane == 0) g.lse[((int64_t)b * g.H + h) * g.T + qi] = mxs + __log2f(sum);
          __syncwarp();
          float a0 = 0.f, a1 = 0.f;
          for (int j = 0; j <= last_key; ++j) {
            float p;
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(p) : "r"(pbuf + 4 * j));
            const float2 vf = bf2_to_f2(lds_u32(sV + sw128_off(j, 2 * lane)));
            a0 += p * vf.x;
            a1 += p * vf.y;
          }
          const float inv = 1.0f / sum;
          const int64_t grow = (int64_t)b * g.T + qi;
          if (g.out)
            *reinterpret_cast<__nv_bfloat162*>(g.out + grow * g.ld_out + h * kTcHd + 2 * lane) =
                __floats2bfloat162_rn(a0 * inv, a1 * inv);
          if (g.out_f32)
            *reinterpret_cast<float2*>(g.out_f32 + grow * g.ld_of + h * kTcHd + 2 * lane) =
                make_float2(a0 * inv, a1 * inv);
          __syncwarp();
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&kv_empty[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTcTmemCols);
}

// host launcher, called from hba_attention_fwd (attention.cu) for bf16 activations
int attention_tc_launch(const __nv_bfloat16* qkv, int64_t ld_qkv, int B, int T, int H, int causal,
                        __nv_bfloat16* out, int64_t ld_out, float* out_f32, int64_t ld_of, float* lse,
                        cudaStream_t stream) {
  static SmemAttr attr;
  HBA_CHECK(ensure_dyn_smem(attention_tc_kernel, kTcSmemBytes, attr, "attention_tc_kernel"));
  AttnTcArgs g;
  g.T = T, g.H = H, g.causal = causal;
  g.n_units = B * H;
  const int rem = T % 128;
  if (T > 128 && rem > 0 && rem <= 8) {
    g.n_tiles = T / 128, g.n_left = rem;
  } else {
    g.n_tiles = (T + 127) / 128, g.n_left = 0;
  }
  if (g.n_tiles > 2) {
    set_error("attention_tc: T=%d needs more than two query tiles", T);
    return HBA_ERR_ARG;
  }
  g.kv_rows = (T + 15) / 16 * 16;
  g.NK = g.kv_rows > 256 ? 256 : g.kv_rows;
  g.n_extra = T > g.NK ? T - g.NK : 0;
  if (g.n_extra > kTcMaxExtra || g.kv_rows > kTcMaxRows) {
    set_error("attention_tc: T=%d exceeds the staged key range", T);
    return HBA_ERR_ARG;
  }
  g.out = out, g.ld_out = ld_out, g.out_f32 = out_f32, g.ld_of = ld_of;
  g.scale_log2 = 1.4426950408889634f * 0.125f;
  g.qkv = qkv, g.ld_qkv = ld_qkv;
  g.lse = lse;
  // [B, T, 3*H*64] maps: the row boxes are rounded up to 16 / 128 rows, and rows >= T of a sequence read
  // as zero instead of the next sequence's (non-finite values there must not reach P = 0 x K / V)
  CUtensorMap t128, t16;
  const uint64_t cols = (uint64_t)3 * H * kTcHd;
  HBA_CHECK(make_tma_3d_bf16(&t128, qkv, B, T, cols, ld_qkv, 128, 64));
  HBA_CHECK(make_tma_3d_bf16(&t16, qkv, B, T, cols, ld_qkv, 16, 64));
  int ctas = num_sms();
  if (g.n_units < ctas) ctas = g.n_units;
  attention_tc_kernel<<<ctas, kTcThreads, kTcSmemBytes, stream>>>(t128, t16, g);
  return check_launch("attention_tc_kernel");
}

}  // namespace hba
