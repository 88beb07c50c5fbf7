// Per-device launch bookkeeping shared by every kernel translation unit (host code only).  What a launch derives from
// its device is cached per device, so that a launch costs at most one cudaGetDevice on top of the launch itself.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace mpe {

constexpr int kCachedDevices = 64;          // ordinals outside [0, 64) are served uncached
constexpr size_t kSmemNoOptIn = 48 * 1024;  // dynamic shared memory every kernel may use without an opt-in

inline int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev;
}

inline int sm_count(int dev) {
  static int cached[kCachedDevices] = {0};
  const bool cache = dev >= 0 && dev < kCachedDevices;
  if (cache && cached[dev] > 0) return cached[dev];
  int n = 0;
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  if (n <= 0) n = 148;  // the B200's count, should the query fail
  if (cache) cached[dev] = n;
  return n;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is sticky per kernel and device: raise it only when a launch needs more
// than was granted before.  The kernel is a template ARGUMENT so that every kernel gets its own record.
template <auto Kernel>
inline cudaError_t ensure_smem(size_t bytes, int dev) {
  if (bytes <= kSmemNoOptIn) return cudaSuccess;
  static size_t granted[kCachedDevices] = {0};
  const bool cache = dev >= 0 && dev < kCachedDevices;
  if (cache && granted[dev] >= bytes) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess && cache) granted[dev] = bytes;
  if (e != cudaSuccess) cudaGetLastError();  // returned here: not left for the next launch's cudaGetLastError
  return e;
}

// For launchers that need the device for nothing else: a request that needs no opt-in does not look it up.
template <auto Kernel>
inline cudaError_t ensure_smem(size_t bytes) {
  return bytes <= kSmemNoOptIn ? cudaSuccess : ensure_smem<Kernel>(bytes, current_device());
}

}  // namespace mpe
