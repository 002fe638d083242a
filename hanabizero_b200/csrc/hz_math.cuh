// Bit-exact float arithmetic for the tree kernels.
//
// The reference tree engine is scalar x86-64 C++ compiled without FMA contraction and calling
// glibc's expf/logf/sqrtf (core/ctree/cnode.cpp:87,385-386).  To give bit-identical priors,
// scores and Q statistics every float operation here is an explicit IEEE round-to-nearest
// intrinsic (__fadd_rn, __fmul_rn, __fdiv_rn, __fsqrt_rn: never contracted into FMA, never
// flushed), and expf is glibc's own algorithm evaluated in fp64:
//   glibc >= 2.27 sysdeps/ieee754/flt-32/e_expf.c + e_exp2f_data.c (N = 32 entry 2^(i/N) table,
//   cubic polynomial), in the evaluation order of the x86-64 ifunc variant selected on any CPU
//   with FMA3 (__expf_fma: the range reduction r = InvLn2N*x - kd is one fused multiply-subtract).
// The host restatement (oracle/expf_glibc.h) is verified against libm for all 2^32 inputs
// (oracle/expf_sweep.c).  Both device copies below are run on the device for all 2^32 inputs and
// compared with that restatement bit for bit (tests/test_device_math_gpu.py; the warp form with 32
// consecutive patterns per warp and with 32 patterns 2^27 apart); tests/test_tree_gpu.py checks the
// kernels' priors bit for bit against the reference.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace hz {

// tab[i] = bits(2^(i/32)) - (i << 47)   (glibc __exp2f_data.tab)
__device__ __constant__ uint64_t k_exp2f_tab[32] = {
    0x3ff0000000000000ull, 0x3fefd9b0d3158574ull, 0x3fefb5586cf9890full, 0x3fef9301d0125b51ull,
    0x3fef72b83c7d517bull, 0x3fef54873168b9aaull, 0x3fef387a6e756238ull, 0x3fef1e9df51fdee1ull,
    0x3fef06fe0a31b715ull, 0x3feef1a7373aa9cbull, 0x3feedea64c123422ull, 0x3feece086061892dull,
    0x3feebfdad5362a27ull, 0x3feeb42b569d4f82ull, 0x3feeab07dd485429ull, 0x3feea47eb03a5585ull,
    0x3feea09e667f3bcdull, 0x3fee9f75e8ec5f74ull, 0x3feea11473eb0187ull, 0x3feea589994cce13ull,
    0x3feeace5422aa0dbull, 0x3feeb737b0cdc5e5ull, 0x3feec49182a3f090ull, 0x3feed503b23e255dull,
    0x3feee89f995ad3adull, 0x3feeff76f2fb5e47ull, 0x3fef199bdd85529cull, 0x3fef3720dcef9069ull,
    0x3fef5818dcfba487ull, 0x3fef7c97337b9b5full, 0x3fefa4afa2a490daull, 0x3fefd0765b6e4540ull,
};

// Warp-cooperative variant: every lane must call.  The 32-entry table is held one entry per lane and
// fetched with two shuffles — a per-lane index into __constant__ memory would serialise into up to 32
// constant-cache replays.
__device__ __forceinline__ float expf_glibc(float x);
__device__ __forceinline__ float expf_glibc_warp(float x, int lane) {
  const double N = 32.0;
  const double InvLn2N = 0x1.71547652b82fep+0 * N;
  const double SHIFT = 0x1.8p+52;
  const double C0 = 0x1.c6af84b912394p-5 / N / N / N;
  const double C1 = 0x1.ebfce50fac4f3p-3 / N / N;
  const double C2 = 0x1.62e42ff0c52d6p-1 / N;
  const uint64_t my_tab = k_exp2f_tab[lane];   // uniform-stride read: one constant-cache pass
  const uint32_t ux = __float_as_uint(x);
  const uint32_t abstop = (ux >> 20) & 0x7ffu;
  const double xd = (double)x;
  const double z = __dmul_rn(InvLn2N, xd);
  double kd = __dadd_rn(z, SHIFT);
  const uint64_t ki = (uint64_t)__double_as_longlong(kd);
  kd = __dsub_rn(kd, SHIFT);
  const double r = __fma_rn(InvLn2N, xd, -kd);
  const int src = (int)(ki & 31u);
  const uint32_t tlo = __shfl_sync(0xffffffffu, (uint32_t)my_tab, src);
  const uint32_t thi = __shfl_sync(0xffffffffu, (uint32_t)(my_tab >> 32), src);
  uint64_t tt = ((uint64_t)thi << 32) | tlo;
  tt += ki << 47;
  const double s = __longlong_as_double((long long)tt);
  const double zz = __dadd_rn(__dmul_rn(C0, r), C1);
  const double r2 = __dmul_rn(r, r);
  double y = __dadd_rn(__dmul_rn(C2, r), 1.0);
  y = __dadd_rn(__dmul_rn(zz, r2), y);
  y = __dmul_rn(y, s);
  float res = __double2float_rn(y);
  if (abstop >= 0x42bu) res = expf_glibc(x);   // |x| >= 88, inf, NaN: the scalar routine's special cases
  return res;
}

__device__ __forceinline__ float expf_glibc(float x) {
  const double N = 32.0;
  const double InvLn2N = 0x1.71547652b82fep+0 * N;
  const double SHIFT = 0x1.8p+52;
  const double C0 = 0x1.c6af84b912394p-5 / N / N / N;
  const double C1 = 0x1.ebfce50fac4f3p-3 / N / N;
  const double C2 = 0x1.62e42ff0c52d6p-1 / N;
  const uint32_t ux = __float_as_uint(x);
  const uint32_t abstop = (ux >> 20) & 0x7ffu;
  if (abstop >= 0x42bu) {  // |x| >= 88 or NaN  (top12(88.0f) = 0x42b)
    if (ux == 0xff800000u) return 0.0f;                    // -inf
    if (abstop >= 0x7f8u) return __fadd_rn(x, x);          // inf / NaN
    if (x > 0x1.62e42ep6f) return __uint_as_float(0x7f800000u);   // overflow
    if (x < -0x1.9fe368p6f) return 0.0f;                           // underflow
    if (x < -0x1.9d1d9ep6f) return __uint_as_float(1u);            // may-underflow: 2^-149
  }
  const double xd = (double)x;
  const double z = __dmul_rn(InvLn2N, xd);
  double kd = __dadd_rn(z, SHIFT);
  const uint64_t ki = (uint64_t)__double_as_longlong(kd);
  kd = __dsub_rn(kd, SHIFT);
  const double r = __fma_rn(InvLn2N, xd, -kd);  // __expf_fma order
  uint64_t t = k_exp2f_tab[ki & 31u];
  t += ki << 47;
  const double s = __longlong_as_double((long long)t);
  const double zz = __dadd_rn(__dmul_rn(C0, r), C1);
  const double r2 = __dmul_rn(r, r);
  double y = __dadd_rn(__dmul_rn(C2, r), 1.0);
  y = __dadd_rn(__dmul_rn(zz, r2), y);
  y = __dmul_rn(y, s);
  return __double2float_rn(y);
}

// monotone float -> uint key (for redux.sync max); NaN must be excluded by the caller
__device__ __forceinline__ uint32_t float_key(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

}  // namespace hz
