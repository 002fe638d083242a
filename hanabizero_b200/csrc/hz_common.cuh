// Shared host/device helpers for libhzb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/hzb200.h"

#define HZ_WARP 32
#define HZ_FULL 0xffffffffu

namespace hz {

void set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_launches;

inline int fail_cuda(cudaError_t e, const char* what) {
  set_error("%s: %s", what, cudaGetErrorString(e));
  return HZ_ERR_CUDA;
}

#define HZ_CUDA(call)                                        \
  do {                                                       \
    cudaError_t _e = (call);                                 \
    if (_e != cudaSuccess) return hz::fail_cuda(_e, #call);  \
  } while (0)

#define HZ_LAUNCH_CHECK(name)                                \
  do {                                                       \
    hz::g_launches.fetch_add(1, std::memory_order_relaxed);  \
    cudaError_t _e = cudaGetLastError();                     \
    if (_e != cudaSuccess) return hz::fail_cuda(_e, name);   \
  } while (0)

// RAII device guard: the handle's device is made current for the call and restored after.
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    target = dev;
  }
  ~DeviceGuard() {
    if (prev >= 0 && prev != target) cudaSetDevice(prev);
  }
  int target = -1;
};

// Non-NULL `p` must be device memory of `device` or page-locked host memory, aligned to `align` bytes.
inline int check_ptr(const char* fn, const char* what, const void* p, int device, int align) {
  if (!p) return HZ_OK;
  if ((uintptr_t)p % align) { set_error("%s: %s must be %d-byte aligned", fn, what, align); return HZ_ERR_ARG; }
  cudaPointerAttributes at{};
  const cudaError_t e = cudaPointerGetAttributes(&at, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail_cuda(e, fn);
  }
  if (at.type == cudaMemoryTypeDevice && at.device == device) return HZ_OK;
  if (at.type == cudaMemoryTypeHost && at.devicePointer == p) return HZ_OK;
  if (at.type == cudaMemoryTypeDevice) {
    set_error("%s: %s is memory of device %d, not of device %d", fn, what, at.device, device);
  } else {
    set_error("%s: %s must be device memory of device %d or page-locked host memory (torch .pin_memory(), "
              "cudaHostAlloc)", fn, what, device);
  }
  return HZ_ERR_ARG;
}

// One root's policy target from its visit counts vc[0, A) (hz_visit_policy, hz_wave_policy): out[a] = vc[a] / sum as a
// correctly rounded double quotient (Python's int / int), all zero when !keep.  out64 / out32 may be NULL.
// A kept row with sum 0 is all NaN (0 / 0, where Python raises); searches leave num_simulations - 1 >= 1 visits.
__device__ __forceinline__ void visit_policy_row(const int32_t* vc, bool keep, int A, double* out64, float* out32) {
  long long sum = 0;   // 32 counts up to 2^31 - 1: past 2^32, exact in 64 bits and in the double it becomes
  for (int a = 0; a < A; ++a) sum += vc[a];
  for (int a = 0; a < A; ++a) {
    // Python: visit_count / sum_visits on ints = correctly rounded double quotient
    const double p = keep ? __ddiv_rn((double)vc[a], (double)sum) : 0.0;
    if (out64) out64[a] = p;
    if (out32) out32[a] = (float)p;
  }
}

}  // namespace hz
