// common.cuh -- error plumbing and small helpers shared by all translation units.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <initializer_list>

namespace nerf {

void set_error(const char* fmt, ...);  // api.cu

#define NERF_CHECK_ARG(cond, ...)            \
  do {                                       \
    if (!(cond)) {                           \
      ::nerf::set_error(__VA_ARGS__);        \
      return -1;                             \
    }                                        \
  } while (0)

#define NERF_CHECK_LAUNCH(name)                                                        \
  do {                                                                                 \
    cudaError_t e__ = cudaGetLastError();                                              \
    if (e__ != cudaSuccess) {                                                          \
      ::nerf::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));       \
      return -2;                                                                       \
    }                                                                                  \
  } while (0)

constexpr int kNumSMs = 148;
constexpr int kMaxDevices = 64;

// Raises the dynamic shared-memory limit of `kernels` to `bytes` on the current device.  The attribute is per device, so
// `done` (one static array per call site) remembers the devices where it has been set.
inline cudaError_t set_max_dynamic_smem_once(bool (&done)[kMaxDevices], std::initializer_list<const void*> kernels, uint32_t bytes) {
  int dev = 0;
  cudaGetDevice(&dev);
  bool& set = done[dev & (kMaxDevices - 1)];
  if (set) return cudaSuccess;
  cudaError_t err = cudaSuccess;
  for (const void* fn : kernels) {
    const cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) err = e;
  }
  set = err == cudaSuccess;
  return err;
}

// ---- flat parameter layout of one NeRFBlock (see include/nerf_b200.h) -----------------
// offsets in floats; every tensor start is padded to a multiple of 4 floats.
struct ParamLayout {
  // initial_layers.{l}.0.weight / bias
  static constexpr int64_t kW0 = 0;                        // 256 x 63
  static constexpr int64_t kB0 = kW0 + 256 * 63;           // 16128
  static constexpr int64_t kW1 = kB0 + 256;                // layers 1..4: 256 x 256 each
  static constexpr int64_t kHiddenStride = 256 * 256 + 256;
  static constexpr int64_t kW5 = kW1 + 4 * kHiddenStride;  // 256 x 319
  static constexpr int64_t kB5 = kW5 + 256 * 319;          // 81664 (multiple of 4)
  static constexpr int64_t kW6 = kB5 + 256;
  static constexpr int64_t kWF = kW6 + 2 * kHiddenStride;  // feature_layer 256 x 256
  static constexpr int64_t kBF = kWF + 256 * 256;
  static constexpr int64_t kWS = kBF + 256;                // density_layer 1 x 256
  static constexpr int64_t kBS = kWS + 256;                // 1 (padded to 4)
  static constexpr int64_t kWC0 = kBS + 4;                 // color_layers.0 128 x 283
  static constexpr int64_t kBC0 = kWC0 + 128 * 283;        // 36224 (multiple of 4)
  static constexpr int64_t kWC1 = kBC0 + 128;              // color_layers.2 3 x 128
  static constexpr int64_t kBC1 = kWC1 + 384;              // 3 (padded to 4)
  static constexpr int64_t kTotal = kBC1 + 4;

  __host__ __device__ static constexpr int64_t hidden_w(int l) {  // l in 0..7
    return l == 0 ? kW0 : (l <= 4 ? kW1 + (l - 1) * kHiddenStride : (l == 5 ? kW5 : kW6 + (l - 6) * kHiddenStride));
  }
  __host__ __device__ static constexpr int64_t hidden_b(int l) {
    return l == 0 ? kB0 : (l <= 4 ? kW1 + (l - 1) * kHiddenStride + 65536 : (l == 5 ? kB5 : kW6 + (l - 6) * kHiddenStride + 65536));
  }
  __host__ __device__ static constexpr int hidden_in(int l) { return l == 0 ? 63 : (l == 5 ? 319 : 256); }
};

// Optional in-kernel stall accounting (tools/kernel_timing.py): when a timing buffer is registered through
// nerf_debug_set_timing(), selected threads accumulate the cycles they spend in each wait and add them to
// the buffer at exit.  A null buffer (the default) costs one predictable branch per wait.
uint64_t* timing_buffer();  // api.cu (host-side registry)
#define NERF_TIMED(enabled, acc, stmt)              \
  do {                                              \
    const long long t0__ = (enabled) ? clock64() : 0; \
    stmt;                                           \
    if (enabled) acc += clock64() - t0__;           \
  } while (0)

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace nerf
