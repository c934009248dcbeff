// Shared helpers for the sm_100a kernels of libhba: error plumbing for the C-ABI, warp
// reductions, and thin inline-PTX wrappers for mbarrier / TMA / tcgen05 / TMEM.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/hba.h"

namespace hba {

// ---- error plumbing (the C-ABI never aborts; it returns a negative code + message) ----
void set_error(const char* fmt, ...);
int check_launch(const char* what);  // 0 or HBA_ERR_CUDA with message

#define HBA_REQUIRE(cond, ...)                  \
  do {                                          \
    if (!(cond)) {                              \
      hba::set_error(__VA_ARGS__);              \
      return HBA_ERR_ARG;                       \
    }                                           \
  } while (0)

constexpr int kNumSMs = 148;
constexpr int kMaxDevices = 64;
int current_device();  // ordinal of the calling thread's current CUDA device (0 when unknown)
int num_sms();         // SM count of the current device (148 on B200)
// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute of a kernel: each launcher keeps one
// SmemAttr (function-local static) and raises the limit on the device it is about to launch on
struct SmemAttr {
  size_t configured[kMaxDevices] = {};
};
template <typename Kernel>
int ensure_dyn_smem(Kernel kernel, size_t bytes, SmemAttr& st, const char* name) {
  const int dev = current_device();
  if (bytes <= st.configured[dev]) return HBA_OK;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("%s: cannot reserve %zu bytes of dynamic shared memory: %s", name, bytes, cudaGetErrorString(e));
    return HBA_ERR_CUDA;
  }
  st.configured[dev] = bytes;
  return HBA_OK;
}
// 2-D bf16 row-major tensor map, box = [box_rows, box_cols]; 64-column boxes use SWIZZLE_128B
int make_tma_2d_bf16(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld,
                     uint32_t box_rows, uint32_t box_cols);
// [batch, rows, cols] bf16 with box [1, box_rows, box_cols]: rows past the end of a batch entry read as zero
int make_tma_3d_bf16(CUtensorMap* map, const void* ptr, uint64_t batch, uint64_t rows, uint64_t cols,
                     uint64_t ld, uint32_t box_rows, uint32_t box_cols);

// pointers a kernel loads / stores as float4 (NULL counts as aligned: optional arguments are checked for presence apart)
inline bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

#define HBA_CHECK(expr)                  \
  do {                                   \
    int _rc = (expr);                    \
    if (_rc != HBA_OK) return _rc;       \
  } while (0)

// ---- warp / block reductions ----
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <typename T>
__device__ __forceinline__ T warp_max(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// block-wide sum, result valid in every thread; `scratch` holds >= 32 T's
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nwarps = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  T r = (lane < nwarps) ? scratch[lane] : T(0);
  return warp_sum(r);
}

// bf16 hi/lo split of an fp32 value: x ~= hi + lo with |x - hi - lo| <= 2^-17 |x|
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// ---- PTX: shared-memory addresses, mbarrier ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// ---- PTX: TMA ----
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tiled load: coordinates are (c0 = innermost element index, c1 = row index)
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0,
                                            int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0,
                                            int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4, %5}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// ---- PTX: tcgen05 / TMEM ----
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 inputs, fp32 accumulate, issued by ONE thread
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets lane (base_lane + t)
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- PTX: CTA pairs (cta_group::2) — two SMs of one TPC run one 256-row UMMA ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// execution-only rendezvous of the cluster (no memory ordering: avoids MEMBAR.ALL.GPU at teardown)
__device__ __forceinline__ void cluster_sync_relaxed() {
  asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
}
// shared::cluster address of `p` (a shared::cta pointer of this CTA) in the CTA of rank `rank`
__device__ __forceinline__ uint32_t mapa_u32(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
// (default .release.cta semantics: an explicit .release.cluster costs MEMBAR.ALL + ERRBAR, i.e. the
// epilogue warp would wait for all its global stores to drain before handing the accumulator back)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr)
               : "memory");
}
// TMA load issued by either CTA of a pair into ITS OWN shared memory; the bytes are accounted on
// the mbarrier at `bar_cluster_addr` (the pair leader's barrier)
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* m,
                                                 uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// 256 x N x 16 UMMA over the pair: each CTA supplies its 128 rows of A and its N/2 rows of B from
// the same shared-memory offsets, and receives its 128 accumulator rows in its own TMEM
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                               uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once the MMAs issued so far have completed) on the barrier at the same offset in every
// CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;" ::"r"(smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}

// UMMA shared-memory matrix descriptor for a K-major bf16 tile stored as rows of 128 bytes with
// the 128-byte swizzle (what a TMA SWIZZLE_128B box of 64 bf16 x R rows produces): 8-row groups are
// 1024 B apart (SBO), LBO is unused for swizzled K-major, descriptor version 1 (Blackwell),
// layout type 2 (SWIZZLE_128B).  Field layout: cute/arch/mma_sm100_desc.hpp `SmemDescriptor`.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);        // start address  [0,14)
  d |= (uint64_t)1 << 16;                         // LBO (ignored)  [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;               // SBO = 1024 B   [32,46)
  d |= (uint64_t)1 << 46;                         // version = 1    [46,48)
  d |= (uint64_t)2 << 61;                         // SWIZZLE_128B   [61,64)
  return d;
}
// Instruction descriptor for kind::f16 with bf16 A/B (both K-major), fp32 D, shape M x N
// (`InstrDescriptor` in cute/arch/mma_sm100_desc.hpp).
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
  return (1u << 4)                   // c_format = F32
         | (1u << 7)                 // a_format = BF16
         | (1u << 10)                // b_format = BF16
         | ((uint32_t)(N >> 3) << 17)  // n_dim
         | ((uint32_t)(M >> 4) << 24); // m_dim
}

}  // namespace hba
