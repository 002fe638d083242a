// TEST INFRASTRUCTURE, not part of libhzb200.so.  Runs the library's own device functions over whole input domains:
//   - glibc's expf, hz_math.cuh's expf_glibc and expf_glibc_warp, over ranges of float bit patterns;
//   - hz_detmath.cuh's det_log and det_exp over arrays of doubles, on the device and, compiled by this same nvcc
//     command, on the host: the host build is the twin the noise kernel's host entry point runs.
// tests/helpers.py:build_detmath_harness compiles it with hanabizero_b200.build.NVCC_FLAGS, so it gets the product's
// -fmad=false -ftz=false -prec-div/-prec-sqrt and host -ffp-contract=off.
#include <cuda_runtime.h>
#include <stdint.h>

#include "hz_detmath.cuh"
#include "hz_math.cuh"

namespace {

// Thread i of a launch evaluates bit pattern start + i, or with `rotate` that index rotated right by 5 bits: lane l
// of a warp then holds (l << 27) | j, so one warp mixes both signs, every exponent range, inf / NaN, the |x| >= 88
// fallback and the polynomial path.
__device__ __forceinline__ uint32_t pattern(uint64_t i, int rotate) {
  const uint32_t u = (uint32_t)i;
  return rotate ? (u >> 5) | (u << 27) : u;
}

__global__ void k_expf(uint32_t* __restrict__ out, uint64_t start, uint64_t n, int rotate) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __float_as_uint(hz::expf_glibc(__uint_as_float(pattern(start + i, rotate))));
}

// n is a multiple of 32, so a warp is either wholly past the end or wholly inside: every lane of a live warp calls
__global__ void k_expf_warp(uint32_t* __restrict__ out, uint64_t start, uint64_t n, int rotate) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = __float_as_uint(hz::expf_glibc_warp(__uint_as_float(pattern(start + i, rotate)), threadIdx.x & 31));
}

__global__ void k_det_log(const double* __restrict__ x, double* __restrict__ y, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = hz::det_log(x[i]);
}

__global__ void k_det_exp(const double* __restrict__ x, double* __restrict__ y, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = hz::det_exp(x[i]);
}

constexpr int kBlock = 256;

unsigned grid(uint64_t n) { return (unsigned)((n + kBlock - 1) / kBlock); }

}  // namespace

extern "C" {
#pragma GCC visibility push(default)

// out[i] = bits of expf_glibc (warp = 0) or expf_glibc_warp (warp = 1) at pattern(start + i, rotate), i < n.
// n must be positive, a multiple of 32, and small enough for a one-dimensional grid.  Returns a cudaError_t.
int hzt_expf(void* stream, uint32_t* out, uint64_t start, uint64_t n, int warp, int rotate) {
  if (n == 0 || n % 32 || grid(n) > 0x7fffffffu) return (int)cudaErrorInvalidValue;
  if (warp)
    k_expf_warp<<<grid(n), kBlock, 0, (cudaStream_t)stream>>>(out, start, n, rotate);
  else
    k_expf<<<grid(n), kBlock, 0, (cudaStream_t)stream>>>(out, start, n, rotate);
  return (int)cudaGetLastError();
}

// y[i] = det_log(x[i]) / det_exp(x[i]) on the device; x and y are device arrays of n doubles
int hzt_det_log(void* stream, const double* x, double* y, int64_t n) {
  if (n <= 0 || grid(n) > 0x7fffffffu) return (int)cudaErrorInvalidValue;
  k_det_log<<<grid(n), kBlock, 0, (cudaStream_t)stream>>>(x, y, n);
  return (int)cudaGetLastError();
}
int hzt_det_exp(void* stream, const double* x, double* y, int64_t n) {
  if (n <= 0 || grid(n) > 0x7fffffffu) return (int)cudaErrorInvalidValue;
  k_det_exp<<<grid(n), kBlock, 0, (cudaStream_t)stream>>>(x, y, n);
  return (int)cudaGetLastError();
}

// the host twin: the same functions compiled for the host; x and y are host arrays of n doubles
void hzt_host_det_log(const double* x, double* y, int64_t n) {
  for (int64_t i = 0; i < n; ++i) y[i] = hz::det_log(x[i]);
}
void hzt_host_det_exp(const double* x, double* y, int64_t n) {
  for (int64_t i = 0; i < n; ++i) y[i] = hz::det_exp(x[i]);
}

#pragma GCC visibility pop
}  // extern "C"
