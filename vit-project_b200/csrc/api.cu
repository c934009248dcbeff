// C-ABI plumbing of libhba: thread-local error message, device check, TMA descriptor encoding.
#include <cstdarg>
#include <cstdio>
#include <mutex>

#include "common.cuh"

namespace hba {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    cudaGetLastError();  // clear the (non-sticky) launch error so that later calls can proceed
    set_error("%s: %s", what, cudaGetErrorString(e));
    return HBA_ERR_CUDA;
  }
  return HBA_OK;
}

int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return (dev >= 0 && dev < kMaxDevices) ? dev : 0;
}

int num_sms() {
  static int cached[kMaxDevices] = {};
  const int dev = current_device();
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      cached[dev] = n;
    else
      return kNumSMs;
  }
  return cached[dev];
}

// cuTensorMapEncodeTiled is resolved through the runtime so that the library has no link-time
// dependency on libcuda (the build container has no driver).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) ==
            cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// 2-D bf16 row-major tensor [rows, cols] with row stride ld (elements); box = [box_rows, 64 cols]
// (64 bf16 = 128 B = one SWIZZLE_128B atom row).  Out-of-bounds elements read as zero.
int make_tma_2d_bf16(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld,
                     uint32_t box_rows, uint32_t box_cols) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is unavailable (no CUDA driver?)");
    return HBA_ERR_CUDA;
  }
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld * 2) % 16 != 0) {
    set_error("TMA operand must be 16-byte aligned with a 16-byte multiple row pitch (ptr=%p ld=%llu)",
              ptr, (unsigned long long)ld);
    return HBA_ERR_ARG;
  }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstr[1] = {ld * 2};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstr, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  box_cols * 2 == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%llu cols=%llu ld=%llu box=%ux%u)",
              (int)r, (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld,
              box_rows, box_cols);
    return HBA_ERR_CUDA;
  }
  return HBA_OK;
}

// 3-D bf16 tensor [batch, rows, cols] (row stride ld elements, batch stride rows * ld) with box
// [1, box_rows, 64 cols]: a box that starts inside one batch entry and runs past its last row reads
// zeros there, never the next entry's first rows.
int make_tma_3d_bf16(CUtensorMap* map, const void* ptr, uint64_t batch, uint64_t rows, uint64_t cols,
                     uint64_t ld, uint32_t box_rows, uint32_t box_cols) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is unavailable (no CUDA driver?)");
    return HBA_ERR_CUDA;
  }
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld * 2) % 16 != 0) {
    set_error("TMA operand must be 16-byte aligned with a 16-byte multiple row pitch (ptr=%p ld=%llu)",
              ptr, (unsigned long long)ld);
    return HBA_ERR_ARG;
  }
  cuuint64_t gdim[3] = {cols, rows, batch};
  cuuint64_t gstr[2] = {ld * 2, rows * ld * 2};
  cuuint32_t box[3] = {box_cols, box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), gdim, gstr, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  box_cols * 2 == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (batch=%llu rows=%llu cols=%llu ld=%llu box=%ux%u)",
              (int)r, (unsigned long long)batch, (unsigned long long)rows, (unsigned long long)cols,
              (unsigned long long)ld, box_rows, box_cols);
    return HBA_ERR_CUDA;
  }
  return HBA_OK;
}

}  // namespace hba

extern "C" {

const char* hba_last_error(void) { return hba::g_err; }

int hba_abi_version(void) { return HBA_ABI_VERSION; }

int hba_device_check(void) {
  int dev = 0, major = 0, minor = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev) != cudaSuccess) {
    cudaGetLastError();
    hba::set_error("no usable CUDA device");
    return HBA_ERR_UNSUPPORTED;
  }
  if (major != 10) {
    hba::set_error("libhba is built for sm_100a only; device is sm_%d%d", major, minor);
    return HBA_ERR_UNSUPPORTED;
  }
  return HBA_OK;
}

}  // extern "C"
