// Root exploration noise on the device with a host twin (SURVEY.md §8f N1).
//
// The reference draws np.random.dirichlet([alpha] * A) per root from numpy's global Mersenne Twister on the host
// (/root/reference/core/selfplay_worker.py:279, reanalyze_worker.py:343) and ships it to C++ through Python lists.
// That stream is sequential (one generator, a variable number of draws per sample), so it cannot be reproduced by
// thousands of roots in parallel.  Here every (root, action) owns a counter-based stream:
//
//   Philox4x32-10 keyed by the 64-bit seed, counter = (block, action, root, step)
//   Gamma(alpha, 1) by Marsaglia & Tsang's method (alpha < 1: Gamma(alpha + 1) * U^(1/alpha)), normals by the
//   polar method, Dirichlet = gammas / their sum (ascending order), rounded once to float32
//
// and — the point of this file — the SAME function runs on the host (hz_host_dirichlet_noise): every floating-point
// operation is an IEEE float64 +, -, *, /, sqrt or fma, and log / exp are fixed polynomials built from those, so the
// host twin returns the device's noise bit for bit (tests/test_noise_gpu.py).  A search can therefore be replayed on
// the CPU — through the reference's own cytree — with exactly the noise the device used.  The twin itself is checked
// against an independent float64 port, Random123's known answers and the float32-rounded Beta law
// (tests/test_noise_reference_cpu.py).
#include <math.h>

#include "hz_common.cuh"

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

// one warp per root on the device
__global__ void __launch_bounds__(128) k_dirichlet(float* __restrict__ out, const float* __restrict__ legal_f32, int N,
                                                   int A, double alpha, unsigned long long seed, uint32_t step,
                                                   uint32_t root_offset) {
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (n >= N) return;
  double g = 0.0, lg = -HUGE_VAL;
  if (lane < A) g = gamma_draw(alpha, seed, step, root_offset + (uint32_t)n, (uint32_t)lane, &lg);
  if (alpha < 1.0) {
    double m = lg;
    for (int o = 16; o > 0; o >>= 1) {
      const double mo = __hiloint2double(__shfl_xor_sync(HZ_FULL, __double2hiint(m), o),
                                         __shfl_xor_sync(HZ_FULL, __double2loint(m), o));
      m = mo > m ? mo : m;
    }
    if (lane < A) g = dirichlet_row_scale(g, lg, m);
  }
  double sum = 0.0;
  for (int a = 0; a < A; ++a) {   // ascending, like numpy's pairwise-free small sums
    const double ga = __hiloint2double(__shfl_sync(HZ_FULL, __double2hiint(g), a), __shfl_sync(HZ_FULL, __double2loint(g), a));
    sum = d_add(sum, ga);
  }
  if (lane < A) {
    float v = (float)d_div(g, sum);
    // reanalyze multiplies the draw by the legal mask (reanalyze_worker.py:343)
    if (legal_f32 && legal_f32[(size_t)n * A + lane] == 0.0f) v = 0.0f;
    out[(size_t)n * A + lane] = v;
  }
}

}  // namespace hz

using namespace hz;

// Finite alpha only, within [1e-300, 1e300]: below, log U / alpha can overflow to -inf for every gamma of a row; above,
// the sum of 32 gammas can overflow to inf.  Both would give NaN rows.
static bool alpha_ok(double alpha) { return alpha >= 1e-300 && alpha <= 1e300; }

extern "C" {
#pragma GCC visibility push(default)

int hz_dirichlet_noise(void* stream, float* out, int num_roots, int num_actions, double alpha, uint64_t seed,
                       uint32_t step, uint32_t root_offset, const float* legal_mask) {
  if (!out || num_roots <= 0 || num_actions <= 0 || num_actions > 32 || !alpha_ok(alpha)) {
    set_error("hz_dirichlet_noise: bad argument");
    return HZ_ERR_ARG;
  }
  k_dirichlet<<<(num_roots + 3) / 4, 128, 0, (cudaStream_t)stream>>>(out, legal_mask, num_roots, num_actions, alpha,
                                                                       seed, step, root_offset);
  HZ_LAUNCH_CHECK("k_dirichlet");
  return HZ_OK;
}

int hz_host_dirichlet_noise(float* out, int num_roots, int num_actions, double alpha, uint64_t seed, uint32_t step,
                            uint32_t root_offset, const float* legal_mask) {
  if (!out || num_roots <= 0 || num_actions <= 0 || num_actions > 32 || !alpha_ok(alpha)) {
    set_error("hz_host_dirichlet_noise: bad argument");
    return HZ_ERR_ARG;
  }
  for (int n = 0; n < num_roots; ++n) {
    double g[32], lg[32], sum = 0.0;
    for (int a = 0; a < num_actions; ++a) {
      lg[a] = -HUGE_VAL;
      g[a] = gamma_draw(alpha, seed, step, root_offset + (uint32_t)n, (uint32_t)a, &lg[a]);
    }
    if (alpha < 1.0) {
      double m = lg[0];
      for (int a = 1; a < num_actions; ++a) m = lg[a] > m ? lg[a] : m;
      for (int a = 0; a < num_actions; ++a) g[a] = dirichlet_row_scale(g[a], lg[a], m);
    }
    for (int a = 0; a < num_actions; ++a) sum = sum + g[a];
    for (int a = 0; a < num_actions; ++a) {
      float v = (float)(g[a] / sum);
      if (legal_mask && legal_mask[(size_t)n * num_actions + a] == 0.0f) v = 0.0f;
      out[(size_t)n * num_actions + a] = v;
    }
  }
  return HZ_OK;
}

#pragma GCC visibility pop
}  // extern "C"
