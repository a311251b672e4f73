// common.cuh -- shared host/device helpers for libsparsifyme_b200.so
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../include/spfy_b200.h"

namespace spfy {

// ---- error reporting: thread-local message, int status --------------------
inline char* err_buf() {
  static thread_local char buf[512] = "";
  return buf;
}
inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(err_buf(), 512, fmt, ap);
  va_end(ap);
  return code;
}
inline std::atomic<uint64_t>& launch_counter() {
  static std::atomic<uint64_t> c{0};
  return c;
}

#define SPFY_CUDA_OK(expr)                                                                  \
  do {                                                                                      \
    cudaError_t e__ = (expr);                                                               \
    if (e__ != cudaSuccess)                                                                 \
      return ::spfy::fail(SPFY_E_CUDA, "%s:%d: %s -> %s", __FILE__, __LINE__, #expr,        \
                          cudaGetErrorString(e__));                                         \
  } while (0)

// call after every kernel launch
#define SPFY_LAUNCH_OK(name)                                                                \
  do {                                                                                      \
    cudaError_t e__ = cudaGetLastError();                                                   \
    if (e__ != cudaSuccess)                                                                 \
      return ::spfy::fail(SPFY_E_CUDA, "launch of %s failed: %s", name,                     \
                          cudaGetErrorString(e__));                                         \
    ::spfy::launch_counter().fetch_add(1, std::memory_order_relaxed);                       \
  } while (0)

// Development switches (ring depth, debug modes that skip work, kernel-choice overrides) are read from the
// environment ONLY in builds made with -DSPFY_DEV_SWITCHES (build.py --dev); the shipped library ignores them,
// so no environment variable can change results or skip work in production.
inline const char* dev_switch(const char* name) {
#ifdef SPFY_DEV_SWITCHES
  return getenv(name);
#else
  (void)name;
  return nullptr;
#endif
}

inline size_t ceil_div(size_t a, size_t b) { return (a + b - 1) / b; }
inline size_t round_up(size_t a, size_t b) { return ceil_div(a, b) * b; }

// device properties are queried once per device and cached
struct DeviceInfo {
  int sm_count = 0;
  int cc_major = 0, cc_minor = 0;
  int max_smem_optin = 0;
};
inline int device_info(DeviceInfo* out) {
  static DeviceInfo cache[64];
  static std::atomic<int> ready[64];
  int dev = 0;
  SPFY_CUDA_OK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return fail(SPFY_E_CUDA, "device index %d out of range", dev);
  if (!ready[dev].load(std::memory_order_acquire)) {
    DeviceInfo d;
    SPFY_CUDA_OK(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev));
    SPFY_CUDA_OK(cudaDeviceGetAttribute(&d.cc_major, cudaDevAttrComputeCapabilityMajor, dev));
    SPFY_CUDA_OK(cudaDeviceGetAttribute(&d.cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
    SPFY_CUDA_OK(cudaDeviceGetAttribute(&d.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    cache[dev] = d;
    ready[dev].store(1, std::memory_order_release);
  }
  *out = cache[dev];
  return SPFY_OK;
}

// the tcgen05 / TMA kernels run on sm_100a only; `di` is filled for the caller
inline int require_sm100(const char* who, DeviceInfo* di) {
  int rc = device_info(di);
  if (rc) return rc;
  if (di->cc_major != 10)
    return fail(SPFY_E_UNSUPPORTED, "%s: needs an sm_100a device, found sm_%d%d", who, di->cc_major, di->cc_minor);
  return SPFY_OK;
}

// grid of a grid-stride kernel: `blocks`, but at most `blocks_per_sm` per SM and at least one
inline int capped_grid(size_t blocks, int blocks_per_sm, int* grid) {
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  *grid = (int)std::max<size_t>(1, std::min(blocks, (size_t)di.sm_count * blocks_per_sm));
  return SPFY_OK;
}

// Raise the dynamic shared-memory limit of `Kernel` to `bytes`: once per device, and again when a call asks for more.
// (Keyed on the kernel itself: different instances of one kernel template share a function type.)
template <auto Kernel>
inline int allow_dynamic_smem(size_t bytes) {
  static std::atomic<size_t> set[64];
  int dev = 0;
  SPFY_CUDA_OK(cudaGetDevice(&dev));
  if (set[dev & 63].load() < bytes) {
    SPFY_CUDA_OK(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    set[dev & 63].store(bytes);
  }
  return SPFY_OK;
}

// ---- element conversion on the device: 16-bit and fp32 to fp32, and back with round-to-nearest-even
__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// SM100 compressed-operand layout (spfy_b200.h): byte offsets, within a value tile (16 KiB) and a metadata tile (2 KiB),
// of the 16-byte value chunk and of the 16-bit metadata word of in-tile row r and 16-column unit q.  (prune.cu spells the
// same sums out inline: in its kernels, folding them into these calls regroups 64-bit address arithmetic and changes
// their SASS.)
__host__ __device__ __forceinline__ uint32_t sm100_val_chunk(uint32_t r, uint32_t q) { return r * 128u + ((q ^ (r & 7u)) << 4); }
__host__ __device__ __forceinline__ uint32_t sm100_meta_word(uint32_t r, uint32_t q) {
  return (r >> 4) * 256u + (q & 1u) * 128u + (r & 7u) * 16u + (q >> 1) * 4u + ((r >> 3) & 1u) * 2u;
}

// The data gradient of a stride-s convolution, split by output phase (spfy_transpose24_conv, spfy_spmma_conv_dgrad).  In
// one spatial dimension of a k-tap filter with padding p, the dx rows ih = s*i + a (0 <= a < s) are
//     dx[s*i + a] = sum over the taps kt = k0, k0 - s, ..., k0 - (taps-1)*s of dy[i + d0 + t] * W[kt],   t = 0, 1, ...
// (dy outside [0, ho) counts as 0): a stride-1 correlation of dy with the phase's taps in descending order.  taps == 0:
// no tap reaches the phase.
struct DgradPhase {
  uint32_t taps;  // taps of the phase
  uint32_t k0;    // its largest filter index
  int d0;         // offset into dy of its first tap (k0): (a + p - k0) / s, exact
};
inline DgradPhase dgrad_phase(size_t k, size_t s, size_t p, size_t a) {
  const size_t r = (a + p) % s;  // the filter indices of phase a are r, r + s, ...
  if (r >= k) return DgradPhase{0u, 0u, 0};
  const size_t k0 = r + (k - 1 - r) / s * s;
  return DgradPhase{(uint32_t)((k0 - r) / s + 1), (uint32_t)k0, ((int)a + (int)p - (int)k0) / (int)s};
}
// dx rows (or columns) of phase a: ceil((h - a) / s)
inline size_t dgrad_phase_extent(size_t h, size_t s, size_t a) { return h > a ? (h - a + s - 1) / s : 0; }

// CUDA loads device code lazily, kernel by kernel, at first use (tens of milliseconds for the big ones).
// Each translation unit lists its kernels here so that spfy_init() can pay that once, outside anybody's timers.
template <typename K>
inline void touch_kernel(K kernel) {
  cudaFuncAttributes a;
  (void)cudaFuncGetAttributes(&a, kernel);
}
void warm_prune_kernels();
void warm_transpose24_kernels();
void warm_spmma_kernels();
void warm_spmm_kernels();
void warm_gemm_kernels();
void warm_optim24_kernels();

inline size_t dtype_bytes(int dtype) {
  switch (dtype) {
    case SPFY_F16:
    case SPFY_BF16: return 2;
    case SPFY_F32: return 4;
    case SPFY_F64: return 8;
    default: return 0;
  }
}

}  // namespace spfy
