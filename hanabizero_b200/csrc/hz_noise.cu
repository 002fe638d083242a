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
// operation is an IEEE float64 +, -, *, /, sqrt or fma, and log / exp are fixed polynomials built from those
// (hz_detmath.cuh), so the host twin returns the device's noise bit for bit.  A search can therefore be replayed on
// the CPU — through the reference's own cytree — with exactly the noise the device used.  Checked by:
//   tests/test_noise_gpu.py          whole rows, device == host, at every A, mask rule and counter edge
//   tests/test_device_math_gpu.py    det_log / det_exp on the device over their whole domain == the host build,
//                                    and whole rows, device == host, across the accepted alpha range [1e-300, 1e300]
//   tests/test_noise_reference_cpu.py  the twin against an independent float64 port, Random123's known answers and
//                                    the float32-rounded Beta law
#include <math.h>

#include "hz_common.cuh"
#include "hz_detmath.cuh"

namespace hz {

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
