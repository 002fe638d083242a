// "Next" rows of the scope table (SURVEY.md §8f N1, N2): the two host hops left between a search and
// the next env step of the self-play loop (/root/reference/core/selfplay_worker.py:258-300).
//   hz_select_action  core/utils.py:280-295 (select_action): drop visits of illegal actions, visit
//                     counts ^ (1/T) -> probabilities, arg-max or inverse-CDF sample
//                     (numpy.random.choice's cdf/searchsorted given the caller's uniform), entropy base 2
//   hz_stack_push     core/game.py:169-174 (GameHistory.step_obs) + selfplay_worker.py:137: the
//                     [N, stack, D] frame stack kept on the device; a finished game's stack is refilled
//                     with the first observation of its next episode
#include <cuda_fp16.h>

#include "hz_common.cuh"

namespace hz {

__global__ void k_select_action(int32_t* __restrict__ visits, const float* __restrict__ legal,
                                const double* __restrict__ temperature, const double* __restrict__ uniforms,
                                int N, int A, int32_t* __restrict__ out_action, float* __restrict__ out_entropy) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  int32_t* v = visits + (size_t)i * A;
  const float* lg = legal + (size_t)i * A;
  const double inv_t = temperature ? 1.0 / temperature[i] : 1.0;   // Python's 1 / temperature, in double
  double p[32];
  double total = 0.0;
  int best = 0, best_v = -2147483647 - 1;
  for (int a = 0; a < A; ++a) {
    int c = v[a];
    if (lg[a] == 0.0f && c >= 1) { c = 0; v[a] = 0; }          // utils.py:282-284 (mutates the counts)
    if (c > best_v) { best_v = c; best = a; }                   // np.argmax: first maximum
    p[a] = (inv_t == 1.0) ? (double)c : pow((double)c, inv_t);  // visit_count ** (1 / temperature)
    total += p[a];                                              // ascending order (not Python >= 3.12's compensated sum)
  }
  if (!(total > 0.0 && isfinite(total))) {
    // no visits left after the zeroing (the reference's ZeroDivisionError), or c^(1/T) or its sum out of range (its
    // OverflowError): no move is defined.  -1 is never legal, so the env kernel raises its sticky illegal-move error.
    out_action[i] = -1;
    if (out_entropy) out_entropy[i] = __int_as_float(0x7fc00000);
    return;
  }
  double ent = 0.0, cum = 0.0;
  for (int a = 0; a < A; ++a) {
    p[a] /= total;
    if (p[a] > 0.0) ent -= p[a] * log(p[a]);                    // scipy.stats.entropy (entr), then / ln 2
  }
  int action = best;
  if (uniforms) {  // np.random.choice: cdf = cumsum(p); cdf /= cdf[-1]; searchsorted(cdf, u, side='right')
    double last = 0.0;
    for (int a = 0; a < A; ++a) last += p[a];
    const double u = uniforms[i];
    action = A - 1;
    for (int a = 0; a < A; ++a) {
      cum += p[a];
      if (u < cum / last) { action = a; break; }
    }
  }
  out_action[i] = action;
  if (out_entropy) out_entropy[i] = (float)(ent / 0.6931471805599453);
}

// one warp per game; stack [N][S][D] floats
__global__ void __launch_bounds__(128) k_stack_push(float* __restrict__ stack, const float* __restrict__ obs,
                                                    int64_t ld_obs, const uint8_t* __restrict__ done, int N, int S,
                                                    int D) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (i >= N) return;
  float* st = stack + (size_t)i * S * D;
  const float* o = obs + (size_t)i * ld_obs;
  const bool refill = done && done[i];
  for (int j = lane; j < D; j += HZ_WARP) {
    const float nv = o[j];
    for (int s = 0; s + 1 < S; ++s) st[(size_t)s * D + j] = refill ? nv : st[(size_t)(s + 1) * D + j];
    st[(size_t)(S - 1) * D + j] = nv;
  }
}

// ---- frame stack as a ring of 0/1 bytes (core/game.py:169-174 without the memmove) --------------------------
// ring [N][S][Dp] uint8 (Dp = frame row padded to 16 bytes; the env kernel writes each new observation straight into
// the slot that holds the oldest frame).  k_ring_gather produces the network input of every game in frame order
// (oldest first): out[i][j * ldf + d] = ring[i][(head + j) % S][d], as half or float, 16 values per lane and step.
template <typename T>
__global__ void __launch_bounds__(128) k_ring_gather(const uint8_t* __restrict__ ring, int head, T* __restrict__ out,
                                                     int64_t ld_out, int ldf, int N, int S, int Dp) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (i >= N) return;
  const int chunks = Dp >> 4;
  for (int j = 0; j < S; ++j) {
    int slot = head + j;
    if (slot >= S) slot -= S;
    const uint4* src = reinterpret_cast<const uint4*>(ring + ((size_t)i * S + slot) * Dp);
    T* dst = out + (size_t)i * ld_out + (size_t)j * ldf;
    for (int c = lane; c < chunks; c += HZ_WARP) {
      const uint4 v = src[c];
      const uint8_t* b = reinterpret_cast<const uint8_t*>(&v);
      if (sizeof(T) == 2) {
        uint4 o0, o1;
        __half2* h0 = reinterpret_cast<__half2*>(&o0);
        __half2* h1 = reinterpret_cast<__half2*>(&o1);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          h0[k] = __floats2half2_rn((float)b[2 * k], (float)b[2 * k + 1]);
          h1[k] = __floats2half2_rn((float)b[8 + 2 * k], (float)b[8 + 2 * k + 1]);
        }
        uint4* d4 = reinterpret_cast<uint4*>(dst + 16 * c);
        d4[0] = o0;
        d4[1] = o1;
      } else {
        float4* d4 = reinterpret_cast<float4*>(dst + 16 * c);
#pragma unroll
        for (int k = 0; k < 4; ++k) d4[k] = make_float4((float)b[4 * k], (float)b[4 * k + 1], (float)b[4 * k + 2], (float)b[4 * k + 3]);
      }
    }
  }
}

// a finished game starts its next episode with the whole stack equal to the first observation (selfplay_worker.py:137)
__global__ void __launch_bounds__(128) k_ring_refill(uint8_t* __restrict__ ring, int src_slot,
                                                     const uint8_t* __restrict__ done, int N, int S, int Dp) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (i >= N || (done && !done[i])) return;
  uint4* base = reinterpret_cast<uint4*>(ring + (size_t)i * S * Dp);
  const int chunks = Dp >> 4;
  for (int c = lane; c < chunks; c += HZ_WARP) {
    const uint4 v = base[(size_t)src_slot * chunks + c];
    for (int s = 0; s < S; ++s)
      if (s != src_slot) base[(size_t)s * chunks + c] = v;
  }
}

}  // namespace hz

using namespace hz;

extern "C" {
#pragma GCC visibility push(default)

int hz_select_action(void* stream, int32_t* visits, const float* legal, const double* temperature,
                     const double* uniforms, int num, int num_actions, int32_t* out_action, float* out_entropy) {
  if (!visits || !legal || !out_action || num <= 0 || num_actions <= 0 || num_actions > 32) {
    set_error("hz_select_action: bad argument");
    return HZ_ERR_ARG;
  }
  k_select_action<<<(num + 127) / 128, 128, 0, (cudaStream_t)stream>>>(visits, legal, temperature, uniforms, num,
                                                                         num_actions, out_action, out_entropy);
  HZ_LAUNCH_CHECK("k_select_action");
  return HZ_OK;
}

int hz_stack_push(void* stream, float* stack, const float* obs, int64_t ld_obs, const uint8_t* done, int num,
                  int stack_depth, int dim) {
  if (!stack || !obs || num <= 0 || stack_depth <= 0 || dim <= 0 || ld_obs < dim) {
    set_error("hz_stack_push: bad argument");
    return HZ_ERR_ARG;
  }
  k_stack_push<<<(num + 3) / 4, 128, 0, (cudaStream_t)stream>>>(stack, obs, ld_obs, done, num, stack_depth, dim);
  HZ_LAUNCH_CHECK("k_stack_push");
  return HZ_OK;
}

int hz_ring_gather(void* stream, const uint8_t* ring, int head, void* out, int64_t ld_out, int frame_stride, int num,
                   int stack_depth, int padded_dim, int elem_bytes) {
  if (!ring || !out || num <= 0 || stack_depth <= 0 || padded_dim <= 0 || (padded_dim & 15) || head < 0 || head >= stack_depth ||
      frame_stride < padded_dim || (frame_stride & 15) || ld_out < (int64_t)stack_depth * frame_stride || (ld_out & 15) ||
      ((uintptr_t)ring & 15) || ((uintptr_t)out & 15) || (elem_bytes != 2 && elem_bytes != 4)) {
    set_error("hz_ring_gather: bad argument (rows and frames must be 16-element aligned)");
    return HZ_ERR_ARG;
  }
  if (elem_bytes == 2) {
    k_ring_gather<__half><<<(num + 3) / 4, 128, 0, (cudaStream_t)stream>>>(ring, head, (__half*)out, ld_out, frame_stride, num,
                                                                          stack_depth, padded_dim);
  } else {
    k_ring_gather<float><<<(num + 3) / 4, 128, 0, (cudaStream_t)stream>>>(ring, head, (float*)out, ld_out, frame_stride, num,
                                                                         stack_depth, padded_dim);
  }
  HZ_LAUNCH_CHECK("k_ring_gather");
  return HZ_OK;
}

int hz_ring_refill(void* stream, uint8_t* ring, int src_slot, const uint8_t* done, int num, int stack_depth, int padded_dim) {
  if (!ring || num <= 0 || stack_depth <= 0 || padded_dim <= 0 || (padded_dim & 15) || src_slot < 0 || src_slot >= stack_depth ||
      ((uintptr_t)ring & 15)) {
    set_error("hz_ring_refill: bad argument");
    return HZ_ERR_ARG;
  }
  k_ring_refill<<<(num + 3) / 4, 128, 0, (cudaStream_t)stream>>>(ring, src_slot, done, num, stack_depth, padded_dim);
  HZ_LAUNCH_CHECK("k_ring_refill");
  return HZ_OK;
}

#pragma GCC visibility pop
}  // extern "C"
