// Float64 primitives of the root noise (hz_noise.cu) that give the same bits on the host and on the device.
//
// Every function here is __host__ __device__ and every floating-point operation is an IEEE float64 +, -, *, /, sqrt or
// fma: the __d*_rn / __fma_rn intrinsics on the device, plain operators and fma() on the host, which the library
// compiles with -ffp-contract=off.  log and exp are fixed polynomials built from those operations, so a gamma draw
// of the device and of its host twin (hz_host_dirichlet_noise) agree bit for bit.  tests/test_device_math_gpu.py
// runs det_log and det_exp on the device over their whole domain against a host build of this header, and
// tests/test_device_math_cpu.py ties that host build to the independent float64 port of
// tests/test_noise_reference_cpu.py.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace hz {

#define HZ_HD __host__ __device__ __forceinline__

HZ_HD double d_mul(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
HZ_HD double d_add(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}
HZ_HD double d_div(double a, double b) {
#ifdef __CUDA_ARCH__
  return __ddiv_rn(a, b);
#else
  return a / b;
#endif
}
HZ_HD double d_sqrt(double a) {
#ifdef __CUDA_ARCH__
  return __dsqrt_rn(a);
#else
  return sqrt(a);
#endif
}
HZ_HD double d_fma(double a, double b, double c) {
#ifdef __CUDA_ARCH__
  return __fma_rn(a, b, c);
#else
  return fma(a, b, c);
#endif
}
HZ_HD unsigned long long d_bits(double x) {
  union { double d; unsigned long long u; } v;
  v.d = x;
  return v.u;
}
HZ_HD double bits_d(unsigned long long u) {
  union { double d; unsigned long long u; } v;
  v.u = u;
  return v.d;
}

// ---- Philox4x32-10 (Salmon et al., SC'11) ---------------------------------------------------------------------
struct Philox4 {
  uint32_t v[4];
};
HZ_HD Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; ++r) {
    const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0, p1 = (unsigned long long)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  Philox4 o;
  o.v[0] = c0; o.v[1] = c1; o.v[2] = c2; o.v[3] = c3;
  return o;
}
// 53 random bits -> a double strictly inside (0, 1): (k + 0.5) * 2^-53, exact
HZ_HD double uniform53(uint32_t hi, uint32_t lo) {
  const unsigned long long k = (((unsigned long long)hi << 32) | lo) >> 11;
  return d_mul(d_add((double)k, 0.5), 1.1102230246251565404236316680908203125e-16);
}

// ---- log and exp from IEEE operations only (identical on host and device; ~1e-15 relative) --------------------
HZ_HD double det_log(double x) {   // x > 0, normal
  unsigned long long b = d_bits(x);
  int e = (int)((b >> 52) & 0x7ff) - 1023;
  double m = bits_d((b & 0x000fffffffffffffull) | 0x3ff0000000000000ull);   // [1, 2)
  if (m > 1.4142135623730951) {
    m = d_mul(m, 0.5);
    e += 1;
  }
  const double s = d_div(d_add(m, -1.0), d_add(m, 1.0)), z = d_mul(s, s);   // log m = 2 atanh(s), |s| <= 0.1716
  double p = 2.0 / 23.0;
  p = d_fma(p, z, 2.0 / 21.0);
  p = d_fma(p, z, 2.0 / 19.0);
  p = d_fma(p, z, 2.0 / 17.0);
  p = d_fma(p, z, 2.0 / 15.0);
  p = d_fma(p, z, 2.0 / 13.0);
  p = d_fma(p, z, 2.0 / 11.0);
  p = d_fma(p, z, 2.0 / 9.0);
  p = d_fma(p, z, 2.0 / 7.0);
  p = d_fma(p, z, 2.0 / 5.0);
  p = d_fma(p, z, 2.0 / 3.0);
  p = d_fma(p, z, 2.0);
  return d_fma((double)e, 0.69314718055994528623, d_mul(s, p));
}
HZ_HD double det_exp(double x) {   // x <= 0
  if (x < -700.0) return 0.0;
  const double kf = floor(d_fma(x, 1.44269504088896338700, 0.5));
  double r = d_fma(kf, -0.693147180369123816490, x);      // ln2 split: high part exact for |k| < 2^10
  r = d_fma(kf, -1.90821492927058770002e-10, r);
  double p = 1.0 / 6227020800.0;   // 1/13!
  p = d_fma(p, r, 1.0 / 479001600.0);
  p = d_fma(p, r, 1.0 / 39916800.0);
  p = d_fma(p, r, 1.0 / 3628800.0);
  p = d_fma(p, r, 1.0 / 362880.0);
  p = d_fma(p, r, 1.0 / 40320.0);
  p = d_fma(p, r, 1.0 / 5040.0);
  p = d_fma(p, r, 1.0 / 720.0);
  p = d_fma(p, r, 1.0 / 120.0);
  p = d_fma(p, r, 1.0 / 24.0);
  p = d_fma(p, r, 1.0 / 6.0);
  p = d_fma(p, r, 0.5);
  p = d_fma(p, r, 1.0);
  p = d_fma(p, r, 1.0);
  const int k = (int)kf;                                   // in [-1010, 0]: the scaling is an exponent add
  return bits_d(d_bits(p) + ((unsigned long long)(long long)k << 52));
}

// Gamma(alpha, 1) of stream (seed, step, root, action).  Every attempt consumes two Philox blocks.  For alpha < 1 the
// draw is d*v * U^(1/alpha), which det_exp cuts to 0 once log U / alpha < -700; *lg receives its logarithm
// log(d*v) + log U / alpha as well, so that a row whose gammas all underflow can be rescaled (dirichlet_row_scale).
HZ_HD double gamma_draw(double alpha, unsigned long long seed, uint32_t step, uint32_t root, uint32_t action,
                        double* lg) {
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const bool boost = alpha < 1.0;
  const double a = boost ? d_add(alpha, 1.0) : alpha;
  const double d = d_add(a, -1.0 / 3.0), c = d_div(1.0, d_sqrt(d_mul(9.0, d)));
  for (uint32_t t = 0;; ++t) {
    const Philox4 b0 = philox4x32_10(2 * t, action, root, step, k0, k1);
    const Philox4 b1 = philox4x32_10(2 * t + 1, action, root, step, k0, k1);
    // polar method: a standard normal from a point of the unit disc
    const double v1 = d_fma(2.0, uniform53(b0.v[0], b0.v[1]), -1.0), v2 = d_fma(2.0, uniform53(b0.v[2], b0.v[3]), -1.0);
    const double s = d_fma(v1, v1, d_mul(v2, v2));
    if (!(s < 1.0) || s == 0.0) continue;
    const double x = d_mul(v1, d_sqrt(d_div(d_mul(-2.0, det_log(s)), s)));
    double v = d_fma(c, x, 1.0);
    if (!(v > 0.0)) continue;
    v = d_mul(d_mul(v, v), v);
    const double u = uniform53(b1.v[0], b1.v[1]);
    const double x2 = d_mul(x, x);
    const bool accept = u < d_fma(-0.0331, d_mul(x2, x2), 1.0) ||
                        det_log(u) < d_fma(0.5, x2, d_mul(d, d_add(d_add(1.0, -v), det_log(v))));
    if (!accept) continue;
    double g = d_mul(d, v);
    if (boost) {   // * U^(1/alpha)
      const double e = d_div(det_log(uniform53(b1.v[2], b1.v[3])), alpha);
      *lg = d_add(det_log(g), e);
      g = d_mul(g, det_exp(e));
    }
    return g;
  }
}

// Row maximum m of the log-gammas (alpha < 1 only).  While m >= -580 the gammas are used as drawn: any of them that
// det_exp cut to 0 (log U / alpha < -700, so lg < -695) is below e^-116 < 2^-150 times the largest and rounds to 0 in
// float32 anyway.  Below, the row is rescaled to exp(lg - m), so its largest gamma is 1 and the sum cannot underflow
// to 0 (a 0/0 row).
HZ_HD double dirichlet_row_scale(double g, double lg, double m) { return m < -580.0 ? det_exp(d_add(lg, -m)) : g; }

}  // namespace hz
