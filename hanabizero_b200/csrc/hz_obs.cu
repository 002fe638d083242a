// Observation tickets (hanabizero_b200/mcts.py, SearchPipeline.submit_observations): the wave's root inference input
// built from stacked observations that the callers hand in as float32 or 0/1 bytes or packed bit strings.
//   hz_obs_pack  every ticket's frames -> rows [k*n, (k+1)*n) of InitialPlan's input x (half or float, frame j at
//                column j * frame_stride, padding columns 0), its legal moves -> the int32 legal staging, its noise ->
//                the noise staging; the rows of unused slots zero (padding roots, as in hz_wave_pack)
//   hz_obs_pack_windows  the same with every obs row a window of stack + positions - 1 consecutive frames: root
//                i * positions + p takes window frames p .. p + stack - 1 (the reanalyze batch, whose consecutive
//                positions share frames, is handed in as one window per sample instead of one stack per position;
//                each root still reads its own stack, so a shared frame is read once per stack that holds it)
//   hz_obs_pack_episodes  the windows read from an episode store's byte arenas (trajectory.EpisodeStore) by
//                (first frame row, last frame row, first legal row, positions with targets) per sample: frames past the
//                episode's end clamped to its last row, legal rows and noise zero and the policy mask 0 past it
// One launch per wave.  The ticket table travels by value in the kernel parameters, as in hz_wave.cu.  Sources are
// device memory or page-locked host memory, read by the kernel itself under unified addressing: for host sources
// the launch is spread over enough CTAs to keep many reads in flight over the host link.
#include <cuda_fp16.h>

#include <algorithm>

#include "hz_common.cuh"

namespace hz {

constexpr int kObsMaxSlots = 64;
constexpr int kObsThreads = 256;
constexpr int kObsChunk = 16;                 // x columns per work item: 16 halves = 2, 16 floats = 4 16-byte stores
constexpr int kObsItemsPerThread = 4;
constexpr int kObsMaxBlocksPerSlot = 1024;
constexpr int kObsMaxStack = 64;
constexpr int kObsMaxCols = 1 << 16;
constexpr int64_t kObsMaxRows = 1 << 24;

struct ObsTable {
  hz_obs_ticket t[kObsMaxSlots];
};
static_assert(sizeof(ObsTable) <= 4096, "the ticket table must fit the kernel parameter space");

struct ObsDims {
  int stack, frame_dim, frame_stride, frame_words, bit_offset, chunks_per_frame, chunks_per_row;
};

// v[0, 16) = src[0, valid), zeros after; 16-byte loads when the whole chunk is there and aligned
__device__ __forceinline__ void load_f32(const float* src, int valid, float* v) {
  if (valid == kObsChunk && ((uintptr_t)src & 15) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(src);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 f = s4[q];
      v[4 * q] = f.x; v[4 * q + 1] = f.y; v[4 * q + 2] = f.z; v[4 * q + 3] = f.w;
    }
  } else {
#pragma unroll
    for (int c = 0; c < kObsChunk; ++c) v[c] = c < valid ? src[c] : 0.f;
  }
}

__device__ __forceinline__ void load_u8(const uint8_t* src, int valid, float* v) {
  if (valid == kObsChunk && ((uintptr_t)src & 15) == 0) {
    const uint4 b = *reinterpret_cast<const uint4*>(src);
    const uint32_t w[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int c = 0; c < kObsChunk; ++c) v[c] = (float)((w[c >> 2] >> (8 * (c & 3))) & 0xffu);
  } else {
#pragma unroll
    for (int c = 0; c < kObsChunk; ++c) v[c] = c < valid ? (float)src[c] : 0.f;
  }
}

// bits [p, p + valid) of the string at `words` (bit b in word b >> 5 at b & 31); valid <= 16, so the chunk spans at most
// two words and is one funnel shift
__device__ __forceinline__ void load_bits(const uint32_t* words, int p, int valid, float* v) {
  uint32_t bits = 0;
  if (valid > 0) {
    const int q = p >> 5, s = p & 31;
    const uint32_t lo = words[q];
    const uint32_t hi = s + valid > 32 ? words[q + 1] : 0u;
    bits = __funnelshift_r(lo, hi, s) & ((1u << valid) - 1u);
  }
#pragma unroll
  for (int c = 0; c < kObsChunk; ++c) v[c] = (float)((bits >> c) & 1u);
}

__device__ __forceinline__ void store_chunk(__half* dst, const float* v) {
  uint4* d4 = reinterpret_cast<uint4*>(dst);
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const __half2 h = __floats2half2_rn(v[8 * q + 2 * e], v[8 * q + 2 * e + 1]);
      w[e] = *reinterpret_cast<const uint32_t*>(&h);
    }
    d4[q] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

__device__ __forceinline__ void store_chunk(float* dst, const float* v) {
  float4* d4 = reinterpret_cast<float4*>(dst);
#pragma unroll
  for (int q = 0; q < 4; ++q) d4[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}

// grid (blocks per slot, slots): blockIdx.y = slot; slots >= count are padding.  Items of a slot: n * chunks_per_row
// 16-column chunks of x (row-major, so neighbouring threads read neighbouring source bytes), then one per row for its
// legal mask and noise.  WIN: root r reads obs row r / positions from frame r % positions on (a compile-time variant,
// so the stack form keeps its own instructions and registers).
template <typename OutT, bool WIN>
__global__ void __launch_bounds__(kObsThreads) k_obs_pack(ObsTable tab, int count, int n, int num_actions, ObsDims d,
                                                          int positions, OutT* __restrict__ x,
                                                          int32_t* __restrict__ legal, float* __restrict__ noise) {
  const int k = blockIdx.y;
  const bool real = k < count;
  // fields read one by one from the parameter space (taking the entry's address would copy the table to local memory)
  const int fmt = real ? tab.t[k].obs_format : -1;
  const char* obs = real ? (const char*)tab.t[k].obs : nullptr;
  const int64_t ld_obs = real ? tab.t[k].ld_obs : 0;
  const int64_t obs_items = (int64_t)n * d.chunks_per_row;
  const int64_t row_cols = (int64_t)d.stack * d.frame_stride;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < obs_items + n; i += stride) {
    if (i < obs_items) {
      const int64_t r = i / d.chunks_per_row;
      const int rem = (int)(i - r * d.chunks_per_row);
      const int j = rem / d.chunks_per_frame;
      const int c0 = (rem - j * d.chunks_per_frame) * kObsChunk;
      const int valid = min(kObsChunk, d.frame_dim - c0);    // <= 0 for a chunk of padding columns only
      int64_t row = r;      // obs row and frame of the source
      int f = j;
      if (WIN) {
        row = r / positions;
        f = j + (int)(r - row * positions);
      }
      float v[kObsChunk];
      if (fmt == HZ_OBS_F32) {
        load_f32((const float*)obs + row * ld_obs + (int64_t)f * d.frame_dim + c0, valid, v);
      } else if (fmt == HZ_OBS_U8) {
        load_u8((const uint8_t*)obs + row * ld_obs + (int64_t)f * d.frame_dim + c0, valid, v);
      } else if (fmt == HZ_OBS_BITS) {
        load_bits((const uint32_t*)obs + row * ld_obs + (int64_t)f * d.frame_words, d.bit_offset + c0, valid, v);
      } else {
#pragma unroll
        for (int c = 0; c < kObsChunk; ++c) v[c] = 0.f;
      }
      store_chunk(x + ((int64_t)k * n + r) * row_cols + (int64_t)j * d.frame_stride + c0, v);
    } else {
      const int64_t r = i - obs_items;
      int32_t* out = legal + ((int64_t)k * n + r) * num_actions;
      const int lfmt = real ? tab.t[k].legal_format : -1;
      const char* src = real ? (const char*)tab.t[k].legal : nullptr;
      const int64_t ld = real ? tab.t[k].ld_legal : 0;
      if (lfmt == HZ_LEGAL_MASK) {
        const uint32_t m = ((const uint32_t*)src)[r * ld];
        for (int a = 0; a < num_actions; ++a) out[a] = (int32_t)((m >> a) & 1u);
      } else if (lfmt == HZ_LEGAL_F32) {
        const float* s = (const float*)src + r * ld;
        for (int a = 0; a < num_actions; ++a) out[a] = s[a] != 0.f ? 1 : 0;
      } else if (lfmt == HZ_LEGAL_I32) {
        const int32_t* s = (const int32_t*)src + r * ld;
        for (int a = 0; a < num_actions; ++a) out[a] = s[a];
      } else {
        for (int a = 0; a < num_actions; ++a) out[a] = 0;
      }
      if (noise) {
        const float* s = real ? tab.t[k].noise : nullptr;
        float* o = noise + ((int64_t)k * n + r) * num_actions;
        for (int a = 0; a < num_actions; ++a) o[a] = s ? s[r * num_actions + a] : 0.f;
      }
    }
  }
}

// Argument checks and the launch of both entry points; positions == 1 without windows is hz_obs_pack.
static int obs_pack(const char* fn, bool windows, void* stream, int device, const hz_obs_ticket* tickets, int count,
                    int slots, int n, int num_actions, const hz_obs_layout* layout, int positions, void* x,
                    int32_t* legal, float* noise) {
  if (!tickets) { set_error("%s: NULL ticket table", fn); return HZ_ERR_ARG; }
  if (!layout) { set_error("%s: NULL layout", fn); return HZ_ERR_ARG; }
  if (slots < 1 || slots > kObsMaxSlots) { set_error("%s: slots = %d, must be 1..%d", fn, slots, kObsMaxSlots); return HZ_ERR_ARG; }
  if (count < 1 || count > slots) { set_error("%s: count = %d, must be 1..slots (%d)", fn, count, slots); return HZ_ERR_ARG; }
  if (n < 1 || (int64_t)slots * n > kObsMaxRows) {
    set_error("%s: n = %d, must be >= 1 with slots * n <= %lld", fn, n, (long long)kObsMaxRows);
    return HZ_ERR_ARG;
  }
  if (positions < 1 || positions > n) { set_error("%s: positions = %d, must be 1..n (%d)", fn, positions, n); return HZ_ERR_ARG; }
  if (n % positions) { set_error("%s: n = %d is not a multiple of positions = %d", fn, n, positions); return HZ_ERR_ARG; }
  if (num_actions < 1 || num_actions > 32) { set_error("%s: num_actions = %d, must be 1..32", fn, num_actions); return HZ_ERR_ARG; }
  const hz_obs_layout L = *layout;
  if (L.stack < 1 || L.stack > kObsMaxStack) { set_error("%s: stack = %d, must be 1..%d", fn, L.stack, kObsMaxStack); return HZ_ERR_ARG; }
  if (L.frame_stride < 16 || L.frame_stride % 16 || (int64_t)L.stack * L.frame_stride > kObsMaxCols) {
    set_error("%s: frame_stride = %d, must be a multiple of 16 with stack * frame_stride <= %d", fn, L.frame_stride, kObsMaxCols);
    return HZ_ERR_ARG;
  }
  if (L.frame_dim < 1 || L.frame_dim > L.frame_stride) {
    set_error("%s: frame_dim = %d, must be 1..frame_stride (%d)", fn, L.frame_dim, L.frame_stride);
    return HZ_ERR_ARG;
  }
  if (L.elem_bytes != 2 && L.elem_bytes != 4) { set_error("%s: elem_bytes = %d, must be 2 or 4", fn, L.elem_bytes); return HZ_ERR_ARG; }
  if (!x || !legal) { set_error("%s: NULL staging buffer", fn); return HZ_ERR_ARG; }
  const int64_t frames = (int64_t)L.stack + positions - 1;     // per obs row: a stack, or a window
  for (int k = 0; k < count; ++k) {
    const hz_obs_ticket& t = tickets[k];
    if (!t.obs || !t.legal) { set_error("%s: ticket %d has a NULL input", fn, k); return HZ_ERR_ARG; }
    if (t.obs_format == HZ_OBS_BITS) {
      if (L.frame_words < 1 || L.bit_offset < 0 || (int64_t)L.bit_offset + L.frame_dim > 32 * (int64_t)L.frame_words) {
        set_error("%s: ticket %d: bit frames need frame_words >= 1 and 0 <= bit_offset, bit_offset + frame_dim <= "
                  "32 * frame_words (frame_words %d, bit_offset %d, frame_dim %d)", fn, k, L.frame_words, L.bit_offset,
                  L.frame_dim);
        return HZ_ERR_ARG;
      }
    } else if (t.obs_format != HZ_OBS_F32 && t.obs_format != HZ_OBS_U8) {
      set_error("%s: ticket %d: obs_format = %d is not a HZ_OBS_* code", fn, k, t.obs_format);
      return HZ_ERR_ARG;
    }
    const int64_t row = frames * (t.obs_format == HZ_OBS_BITS ? L.frame_words : L.frame_dim);
    if (t.ld_obs < row) {
      set_error("%s: ticket %d: ld_obs = %lld, must be >= the %lld elements of a %s", fn, k, (long long)t.ld_obs,
                (long long)row, windows ? "window" : "row");
      return HZ_ERR_ARG;
    }
    if (t.legal_format != HZ_LEGAL_I32 && t.legal_format != HZ_LEGAL_F32 && t.legal_format != HZ_LEGAL_MASK) {
      set_error("%s: ticket %d: legal_format = %d is not a HZ_LEGAL_* code", fn, k, t.legal_format);
      return HZ_ERR_ARG;
    }
    const int64_t lrow = t.legal_format == HZ_LEGAL_MASK ? 1 : num_actions;
    if (t.ld_legal < lrow) {
      set_error("%s: ticket %d: ld_legal = %lld, must be >= %lld", fn, k, (long long)t.ld_legal, (long long)lrow);
      return HZ_ERR_ARG;
    }
  }
  DeviceGuard dg(device);
  if (!dg.ok) return fail_cuda(cudaGetLastError(), fn);
  if (int rc = check_ptr(fn, "staging x", x, device, 16)) return rc;
  if (int rc = check_ptr(fn, "staging legal", legal, device, 4)) return rc;
  if (int rc = check_ptr(fn, "staging noise", noise, device, 4)) return rc;
  for (int k = 0; k < count; ++k) {
    const hz_obs_ticket& t = tickets[k];
    if (int rc = check_ptr(fn, "ticket obs", t.obs, device, t.obs_format == HZ_OBS_U8 ? 1 : 4)) return rc;
    if (int rc = check_ptr(fn, "ticket legal", t.legal, device, 4)) return rc;
    if (int rc = check_ptr(fn, "ticket noise", t.noise, device, 4)) return rc;
  }
  ObsTable tab{};
  for (int k = 0; k < count; ++k) tab.t[k] = tickets[k];
  ObsDims d;
  d.stack = L.stack, d.frame_dim = L.frame_dim, d.frame_stride = L.frame_stride, d.frame_words = L.frame_words;
  d.bit_offset = L.bit_offset, d.chunks_per_frame = L.frame_stride / kObsChunk;
  d.chunks_per_row = L.stack * d.chunks_per_frame;
  const int64_t items = (int64_t)n * (d.chunks_per_row + 1);
  const int64_t per_block = (int64_t)kObsThreads * kObsItemsPerThread;
  const int blocks = (int)std::min<int64_t>((items + per_block - 1) / per_block, kObsMaxBlocksPerSlot);
  const dim3 grid(blocks, slots);
  cudaStream_t st = (cudaStream_t)stream;
  if (windows) {
    if (L.elem_bytes == 2) {
      k_obs_pack<__half, true><<<grid, kObsThreads, 0, st>>>(tab, count, n, num_actions, d, positions, (__half*)x, legal, noise);
    } else {
      k_obs_pack<float, true><<<grid, kObsThreads, 0, st>>>(tab, count, n, num_actions, d, positions, (float*)x, legal, noise);
    }
    HZ_LAUNCH_CHECK("k_obs_pack<windows>");
  } else {
    if (L.elem_bytes == 2) {
      k_obs_pack<__half, false><<<grid, kObsThreads, 0, st>>>(tab, count, n, num_actions, d, 1, (__half*)x, legal, noise);
    } else {
      k_obs_pack<float, false><<<grid, kObsThreads, 0, st>>>(tab, count, n, num_actions, d, 1, (float*)x, legal, noise);
    }
    HZ_LAUNCH_CHECK("k_obs_pack");
  }
  return HZ_OK;
}

// ---- episode tickets: windows read straight from an episode store's arenas ------------------------------------------

struct EpisodeTable {
  hz_obs_episode_ticket t[kObsMaxSlots];
};
static_assert(sizeof(EpisodeTable) <= 4096, "the ticket table must fit the kernel parameter space");

// grid and items as k_obs_pack<OutT, true>.  Root r = i * positions + p of a ticket reads its frames j = 0..stack-1 from
// arena row min(first + p + j, last) of sample i, and its legal row, noise and mask from the sample's target count.
template <typename OutT>
__global__ void __launch_bounds__(kObsThreads) k_obs_pack_episodes(EpisodeTable tab, int count, int n, int num_actions,
                                                                   ObsDims d, int positions, OutT* __restrict__ x,
                                                                   int32_t* __restrict__ legal,
                                                                   float* __restrict__ noise) {
  const int k = blockIdx.y;
  const bool real = k < count;
  const uint8_t* frames = real ? tab.t[k].frames : nullptr;
  const int64_t ld = real ? tab.t[k].ld_frames : 0;
  const int32_t* samples = real ? tab.t[k].samples : nullptr;
  const int64_t obs_items = (int64_t)n * d.chunks_per_row;
  const int64_t row_cols = (int64_t)d.stack * d.frame_stride;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < obs_items + n; i += stride) {
    if (i < obs_items) {
      const int64_t r = i / d.chunks_per_row;
      const int rem = (int)(i - r * d.chunks_per_row);
      const int j = rem / d.chunks_per_frame;
      const int c0 = (rem - j * d.chunks_per_frame) * kObsChunk;
      const int valid = min(kObsChunk, d.frame_dim - c0);
      float v[kObsChunk];
      if (real) {
        const int64_t s = r / positions;
        const int p = (int)(r - s * positions);
        const int4 smp = reinterpret_cast<const int4*>(samples)[s];
        const int64_t row = min(smp.x + p + j, smp.y);
        load_u8(frames + row * ld + c0, valid, v);
      } else {
#pragma unroll
        for (int c = 0; c < kObsChunk; ++c) v[c] = 0.f;
      }
      store_chunk(x + ((int64_t)k * n + r) * row_cols + (int64_t)j * d.frame_stride + c0, v);
    } else {
      const int64_t r = i - obs_items;
      int32_t* out = legal + ((int64_t)k * n + r) * num_actions;
      float* o = noise ? noise + ((int64_t)k * n + r) * num_actions : nullptr;
      const uint8_t* src = nullptr;
      if (real) {
        const int64_t s = r / positions;
        const int p = (int)(r - s * positions);
        const int4 smp = reinterpret_cast<const int4*>(samples)[s];
        const bool keep = p < smp.w;
        if (keep) src = tab.t[k].legal + (int64_t)(smp.z + p) * num_actions;
        tab.t[k].mask[r] = keep ? 1 : 0;
      }
      const float* nz = real ? tab.t[k].noise : nullptr;
      for (int a = 0; a < num_actions; ++a) {
        const bool on = src && src[a] != 0;
        out[a] = on ? 1 : 0;
        if (o) o[a] = on && nz ? nz[r * num_actions + a] : 0.f;
      }
    }
  }
}

static int obs_pack_episodes(const char* fn, void* stream, int device, const hz_obs_episode_ticket* tickets, int count,
                             int slots, int n, int num_actions, const hz_obs_layout* layout, int positions, void* x,
                             int32_t* legal, float* noise) {
  if (!tickets) { set_error("%s: NULL ticket table", fn); return HZ_ERR_ARG; }
  if (!layout) { set_error("%s: NULL layout", fn); return HZ_ERR_ARG; }
  if (slots < 1 || slots > kObsMaxSlots) { set_error("%s: slots = %d, must be 1..%d", fn, slots, kObsMaxSlots); return HZ_ERR_ARG; }
  if (count < 1 || count > slots) { set_error("%s: count = %d, must be 1..slots (%d)", fn, count, slots); return HZ_ERR_ARG; }
  if (n < 1 || (int64_t)slots * n > kObsMaxRows) {
    set_error("%s: n = %d, must be >= 1 with slots * n <= %lld", fn, n, (long long)kObsMaxRows);
    return HZ_ERR_ARG;
  }
  if (positions < 1 || positions > n) { set_error("%s: positions = %d, must be 1..n (%d)", fn, positions, n); return HZ_ERR_ARG; }
  if (n % positions) { set_error("%s: n = %d is not a multiple of positions = %d", fn, n, positions); return HZ_ERR_ARG; }
  if (num_actions < 1 || num_actions > 32) { set_error("%s: num_actions = %d, must be 1..32", fn, num_actions); return HZ_ERR_ARG; }
  const hz_obs_layout L = *layout;
  if (L.stack < 1 || L.stack > kObsMaxStack) { set_error("%s: stack = %d, must be 1..%d", fn, L.stack, kObsMaxStack); return HZ_ERR_ARG; }
  if (L.frame_stride < 16 || L.frame_stride % 16 || (int64_t)L.stack * L.frame_stride > kObsMaxCols) {
    set_error("%s: frame_stride = %d, must be a multiple of 16 with stack * frame_stride <= %d", fn, L.frame_stride, kObsMaxCols);
    return HZ_ERR_ARG;
  }
  if (L.frame_dim < 1 || L.frame_dim > L.frame_stride) {
    set_error("%s: frame_dim = %d, must be 1..frame_stride (%d)", fn, L.frame_dim, L.frame_stride);
    return HZ_ERR_ARG;
  }
  if (L.elem_bytes != 2 && L.elem_bytes != 4) { set_error("%s: elem_bytes = %d, must be 2 or 4", fn, L.elem_bytes); return HZ_ERR_ARG; }
  if (!x || !legal) { set_error("%s: NULL staging buffer", fn); return HZ_ERR_ARG; }
  for (int k = 0; k < count; ++k) {
    const hz_obs_episode_ticket& t = tickets[k];
    if (!t.frames || !t.legal || !t.samples) { set_error("%s: ticket %d has a NULL input", fn, k); return HZ_ERR_ARG; }
    if (!t.mask) { set_error("%s: ticket %d has a NULL mask output", fn, k); return HZ_ERR_ARG; }
    if (t.ld_frames < L.frame_dim) {
      set_error("%s: ticket %d: ld_frames = %lld, must be >= frame_dim (%d)", fn, k, (long long)t.ld_frames, L.frame_dim);
      return HZ_ERR_ARG;
    }
  }
  DeviceGuard dg(device);
  if (!dg.ok) return fail_cuda(cudaGetLastError(), fn);
  if (int rc = check_ptr(fn, "staging x", x, device, 16)) return rc;
  if (int rc = check_ptr(fn, "staging legal", legal, device, 4)) return rc;
  if (int rc = check_ptr(fn, "staging noise", noise, device, 4)) return rc;
  for (int k = 0; k < count; ++k) {
    const hz_obs_episode_ticket& t = tickets[k];
    if (int rc = check_ptr(fn, "ticket frames", t.frames, device, 1)) return rc;
    if (int rc = check_ptr(fn, "ticket legal", t.legal, device, 1)) return rc;
    if (int rc = check_ptr(fn, "ticket samples", t.samples, device, 16)) return rc;
    if (int rc = check_ptr(fn, "ticket noise", t.noise, device, 4)) return rc;
    if (int rc = check_ptr(fn, "ticket mask", t.mask, device, 1)) return rc;
  }
  EpisodeTable tab{};
  for (int k = 0; k < count; ++k) tab.t[k] = tickets[k];
  ObsDims d;
  d.stack = L.stack, d.frame_dim = L.frame_dim, d.frame_stride = L.frame_stride, d.frame_words = L.frame_words;
  d.bit_offset = L.bit_offset, d.chunks_per_frame = L.frame_stride / kObsChunk;
  d.chunks_per_row = L.stack * d.chunks_per_frame;
  const int64_t items = (int64_t)n * (d.chunks_per_row + 1);
  const int64_t per_block = (int64_t)kObsThreads * kObsItemsPerThread;
  const int blocks = (int)std::min<int64_t>((items + per_block - 1) / per_block, kObsMaxBlocksPerSlot);
  const dim3 grid(blocks, slots);
  cudaStream_t st = (cudaStream_t)stream;
  if (L.elem_bytes == 2) {
    k_obs_pack_episodes<__half><<<grid, kObsThreads, 0, st>>>(tab, count, n, num_actions, d, positions, (__half*)x, legal, noise);
  } else {
    k_obs_pack_episodes<float><<<grid, kObsThreads, 0, st>>>(tab, count, n, num_actions, d, positions, (float*)x, legal, noise);
  }
  HZ_LAUNCH_CHECK("k_obs_pack_episodes");
  return HZ_OK;
}

}  // namespace hz

using namespace hz;

extern "C" {
#pragma GCC visibility push(default)

int hz_obs_pack(void* stream, int device, const hz_obs_ticket* tickets, int count, int slots, int n, int num_actions,
                const hz_obs_layout* layout, void* x, int32_t* legal, float* noise) {
  return obs_pack("hz_obs_pack", false, stream, device, tickets, count, slots, n, num_actions, layout, 1, x, legal, noise);
}

int hz_obs_pack_windows(void* stream, int device, const hz_obs_ticket* tickets, int count, int slots, int n,
                        int num_actions, const hz_obs_layout* layout, int positions, void* x, int32_t* legal,
                        float* noise) {
  return obs_pack("hz_obs_pack_windows", true, stream, device, tickets, count, slots, n, num_actions, layout, positions,
                  x, legal, noise);
}

int hz_obs_pack_episodes(void* stream, int device, const hz_obs_episode_ticket* tickets, int count, int slots, int n,
                         int num_actions, const hz_obs_layout* layout, int positions, void* x, int32_t* legal,
                         float* noise) {
  return obs_pack_episodes("hz_obs_pack_episodes", stream, device, tickets, count, slots, n, num_actions, layout,
                           positions, x, legal, noise);
}

#pragma GCC visibility pop
}  // extern "C"
