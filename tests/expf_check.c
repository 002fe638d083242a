/* TEST INFRASTRUCTURE.  Host reference of the device expf sweep (tests/test_device_math_gpu.py): device outputs over a
 * range of float bit patterns against the glibc restatement hz_expf_glibc(x, 1) of oracle/expf_glibc.h, which
 * tests/test_oracle_expf.py and oracle/expf_sweep.c tie to libm.  Built the way expf_sweep.c is:
 *   gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC -I oracle expf_check.c -lm */
#include <stdlib.h>

#include "expf_glibc.h"

/* the pattern of index i: tests/detmath_harness.cu's pattern() */
static inline uint32_t pattern(uint64_t i, int rotate) {
  const uint32_t u = (uint32_t)i;
  return rotate ? (u >> 5) | (u << 27) : u;
}

enum { BLOCKS = 256 };

/* outs[k][i] (k < nout, i < n) holds the bits the device returned for pattern(start + i, rotate).  It must equal
 * hz_expf_glibc bit for bit, except that a NaN result only has to be a NaN (payloads are not part of the contract).
 * bad[k] receives the number of mismatches of output k, first[k * nfirst ...] its first min(bad[k], nfirst)
 * mismatching patterns in index order.  Returns -1 if it cannot allocate, else 0. */
int hz_expf_check(const uint32_t* const* outs, int nout, uint64_t start, uint64_t n, int rotate, uint64_t* bad,
                  uint32_t* first, int nfirst) {
  uint64_t* cnt = calloc((size_t)BLOCKS * nout, sizeof(uint64_t));
  uint32_t* pat = calloc((size_t)BLOCKS * nout * (nfirst > 0 ? nfirst : 1), sizeof(uint32_t));
  if (!cnt || !pat) {
    free(cnt);
    free(pat);
    return -1;
  }
#pragma omp parallel for schedule(dynamic)
  for (int b = 0; b < BLOCKS; ++b) {
    const uint64_t lo = n * b / BLOCKS, hi = n * (b + 1) / BLOCKS;
    for (uint64_t i = lo; i < hi; ++i) {
      const uint32_t p = pattern(start + i, rotate);
      float x;
      memcpy(&x, &p, 4);
      const float ref = hz_expf_glibc(x, 1);
      const int refnan = ref != ref;
      const uint32_t rb = hz_asuint(ref);
      for (int k = 0; k < nout; ++k) {
        const uint32_t d = outs[k][i];
        const int dnan = (d & 0x7f800000u) == 0x7f800000u && (d & 0x007fffffu);
        if (refnan ? dnan : d == rb) continue;
        uint64_t* c = &cnt[(size_t)b * nout + k];
        if (*c < (uint64_t)nfirst) pat[((size_t)b * nout + k) * nfirst + *c] = p;
        ++*c;
      }
    }
  }
  for (int k = 0; k < nout; ++k) {
    uint64_t total = 0;
    for (int b = 0; b < BLOCKS; ++b) {
      const uint64_t c = cnt[(size_t)b * nout + k];
      for (uint64_t j = 0; j < c && j < (uint64_t)nfirst && total + j < (uint64_t)nfirst; ++j)
        first[(size_t)k * nfirst + total + j] = pat[((size_t)b * nout + k) * nfirst + j];
      total += c;
    }
    bad[k] = total;
  }
  free(cnt);
  free(pat);
  return 0;
}
