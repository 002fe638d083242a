// Search waves (hanabizero_b200/mcts.py, SearchPipeline(wave=G)): G independent root batches ("tickets") of n roots
// each are searched as one batch of G*n trees.  Trees never interact, so the wave only needs its inputs gathered into
// one set of staging buffers and its root statistics scattered back:
//   hz_wave_pack    every ticket's prepare inputs and root hidden states -> rows [k*n, (k+1)*n) of the staging
//                   buffers, the rows of unused slots zero-filled (all-zero legal mask: a root without children)
//   hz_wave_unpack  rows [k*n, (k+1)*n) of the wave's statistics buffer -> ticket k's outputs
//   hz_wave_policy  the visit counts of the same rows -> ticket k's float64 policy targets (hz_visit_policy's
//                   arithmetic, per ticket mask)
// One launch each, in place of 5*G + 2*G cudaMemcpyAsync calls.  The ticket table travels by value in the kernel
// parameters (64 x 56 B), so no descriptor buffer has to be updated in stream order.  Sources and destinations are
// device memory or page-locked host memory, which the kernel reads and writes itself under unified addressing (as
// hz_envs_host_step does).
#include "hz_common.cuh"

namespace hz {

constexpr int kWaveMaxSlots = 64;
constexpr int kWaveThreads = 256;
constexpr int kWaveBlocksPerSlot = 16;
constexpr int64_t kWaveMaxRows = 1 << 24;
constexpr int kWaveMaxRowBytes = 1 << 16;

struct WaveTable {
  hz_wave_ticket t[kWaveMaxSlots];
};
static_assert(sizeof(WaveTable) <= 4096, "the ticket table must fit the kernel parameter space");

struct PolicyTable {
  hz_policy_ticket t[kWaveMaxSlots];
};
static_assert(sizeof(PolicyTable) == 64 * 16, "the policy table is 64 x 16 B of kernel parameters");
constexpr int kPolicyThreads = 128;

// dst[0, words) = src[0, words), or zeros when src == NULL; 16-byte vectors when both ends allow, 4-byte words
// otherwise.  The calling slot's blocks split the range.
__device__ __forceinline__ void copy_words(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, int64_t words) {
  const int64_t lane = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  if ((((uintptr_t)dst | (uintptr_t)src) & 15) == 0) {
    const int64_t vecs = words >> 2;
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    for (int64_t i = lane; i < vecs; i += stride) d4[i] = src ? s4[i] : make_uint4(0, 0, 0, 0);
    for (int64_t i = (vecs << 2) + lane; i < words; i += stride) dst[i] = src ? src[i] : 0u;
  } else {
    for (int64_t i = lane; i < words; i += stride) dst[i] = src ? src[i] : 0u;
  }
}

// grid (kWaveBlocksPerSlot, slots): blockIdx.y = slot; slots >= count are padding
__global__ void __launch_bounds__(kWaveThreads) k_wave_pack(WaveTable tab, int count, int n, int num_actions,
                                                            int row_words, uint32_t* noise, uint32_t* reward,
                                                            uint32_t* logits, uint32_t* legal, uint32_t* hidden) {
  const int k = blockIdx.y;
  const bool real = k < count;
  // fields read one by one from the parameter space (taking the entry's address would copy the table to local memory)
  const uint32_t* s_noise = real ? (const uint32_t*)tab.t[k].noise : nullptr;
  const uint32_t* s_reward = real ? (const uint32_t*)tab.t[k].reward : nullptr;
  const uint32_t* s_logits = real ? (const uint32_t*)tab.t[k].logits : nullptr;
  const uint32_t* s_legal = real ? (const uint32_t*)tab.t[k].legal : nullptr;
  const uint32_t* s_hidden = real ? (const uint32_t*)tab.t[k].hidden : nullptr;
  const int64_t na = (int64_t)n * num_actions;
  if (noise) copy_words(noise + k * na, s_noise, na);
  copy_words(reward + (int64_t)k * n, s_reward, n);
  copy_words(logits + k * na, s_logits, na);
  copy_words(legal + k * na, s_legal, na);
  copy_words(hidden + (int64_t)k * n * row_words, s_hidden, (int64_t)n * row_words);
}

// grid (kWaveBlocksPerSlot, count)
__global__ void __launch_bounds__(kWaveThreads) k_wave_unpack(WaveTable tab, int slots, int n, int num_actions,
                                                              const uint32_t* stats) {
  const int k = blockIdx.y;
  const int64_t na = (int64_t)n * num_actions;
  if (tab.t[k].out_visits) copy_words((uint32_t*)tab.t[k].out_visits, stats + k * na, na);
  if (tab.t[k].out_values) copy_words((uint32_t*)tab.t[k].out_values, stats + slots * na + (int64_t)k * n, n);
}

// grid (ceil(n / kPolicyThreads), count): one thread per root of ticket blockIdx.y
__global__ void __launch_bounds__(kPolicyThreads) k_wave_policy(PolicyTable tab, int n, int num_actions,
                                                                const int32_t* __restrict__ stats) {
  const int k = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint8_t* mask = tab.t[k].mask;
  visit_policy_row(stats + ((int64_t)k * n + i) * num_actions, !mask || mask[i], num_actions,
                   tab.t[k].out + (int64_t)i * num_actions, nullptr);
}

static int check_sizes(const char* fn, const hz_wave_ticket* tickets, int count, int slots, int n, int num_actions) {
  if (!tickets) { set_error("%s: NULL ticket table", fn); return HZ_ERR_ARG; }
  if (slots < 1 || slots > kWaveMaxSlots) { set_error("%s: slots = %d, must be 1..%d", fn, slots, kWaveMaxSlots); return HZ_ERR_ARG; }
  if (count < 1 || count > slots) { set_error("%s: count = %d, must be 1..slots (%d)", fn, count, slots); return HZ_ERR_ARG; }
  if (n < 1 || (int64_t)slots * n > kWaveMaxRows) {
    set_error("%s: n = %d, must be >= 1 with slots * n <= %lld", fn, n, (long long)kWaveMaxRows);
    return HZ_ERR_ARG;
  }
  if (num_actions < 1 || num_actions > 32) { set_error("%s: num_actions = %d, must be 1..32", fn, num_actions); return HZ_ERR_ARG; }
  return HZ_OK;
}

}  // namespace hz

using namespace hz;

extern "C" {
#pragma GCC visibility push(default)

int hz_wave_pack(void* stream, int device, const hz_wave_ticket* tickets, int count, int slots, int n, int num_actions,
                 int hidden_row_bytes, float* noise, float* reward, float* logits, int32_t* legal, void* hidden) {
  const char* fn = "hz_wave_pack";
  if (int rc = check_sizes(fn, tickets, count, slots, n, num_actions)) return rc;
  if (hidden_row_bytes < 16 || hidden_row_bytes > kWaveMaxRowBytes || hidden_row_bytes % 16) {
    set_error("%s: hidden_row_bytes = %d, must be a multiple of 16 in 16..%d", fn, hidden_row_bytes, kWaveMaxRowBytes);
    return HZ_ERR_ARG;
  }
  if (!reward || !logits || !legal || !hidden) { set_error("%s: NULL staging buffer", fn); return HZ_ERR_ARG; }
  for (int k = 0; k < count; ++k) {
    if (!tickets[k].reward || !tickets[k].logits || !tickets[k].legal || !tickets[k].hidden) {
      set_error("%s: ticket %d has a NULL input", fn, k);
      return HZ_ERR_ARG;
    }
  }
  DeviceGuard dg(device);
  if (!dg.ok) return fail_cuda(cudaGetLastError(), fn);
  const struct { const char* what; const void* p; int align; } staging[5] = {
      {"staging noise", noise, 4}, {"staging reward", reward, 4}, {"staging logits", logits, 4},
      {"staging legal", legal, 4}, {"staging hidden", hidden, 16}};
  for (const auto& s : staging) {
    if (int rc = check_ptr(fn, s.what, s.p, device, s.align)) return rc;
  }
  for (int k = 0; k < count; ++k) {
    const hz_wave_ticket& t = tickets[k];
    if (int rc = check_ptr(fn, "ticket noise", t.noise, device, 4)) return rc;
    if (int rc = check_ptr(fn, "ticket reward", t.reward, device, 4)) return rc;
    if (int rc = check_ptr(fn, "ticket logits", t.logits, device, 4)) return rc;
    if (int rc = check_ptr(fn, "ticket legal", t.legal, device, 4)) return rc;
    if (int rc = check_ptr(fn, "ticket hidden", t.hidden, device, 16)) return rc;
  }
  WaveTable tab{};
  for (int k = 0; k < count; ++k) tab.t[k] = tickets[k];
  k_wave_pack<<<dim3(kWaveBlocksPerSlot, slots), kWaveThreads, 0, (cudaStream_t)stream>>>(
      tab, count, n, num_actions, hidden_row_bytes / 4, (uint32_t*)noise, (uint32_t*)reward, (uint32_t*)logits,
      (uint32_t*)legal, (uint32_t*)hidden);
  HZ_LAUNCH_CHECK("k_wave_pack");
  return HZ_OK;
}

int hz_wave_unpack(void* stream, int device, const hz_wave_ticket* tickets, int count, int slots, int n,
                   int num_actions, const int32_t* stats) {
  const char* fn = "hz_wave_unpack";
  if (int rc = check_sizes(fn, tickets, count, slots, n, num_actions)) return rc;
  if (!stats) { set_error("%s: NULL statistics buffer", fn); return HZ_ERR_ARG; }
  DeviceGuard dg(device);
  if (!dg.ok) return fail_cuda(cudaGetLastError(), fn);
  if (int rc = check_ptr(fn, "statistics buffer", stats, device, 4)) return rc;
  for (int k = 0; k < count; ++k) {
    if (int rc = check_ptr(fn, "ticket out_visits", tickets[k].out_visits, device, 4)) return rc;
    if (int rc = check_ptr(fn, "ticket out_values", tickets[k].out_values, device, 4)) return rc;
  }
  WaveTable tab{};
  for (int k = 0; k < count; ++k) tab.t[k] = tickets[k];
  k_wave_unpack<<<dim3(kWaveBlocksPerSlot, count), kWaveThreads, 0, (cudaStream_t)stream>>>(
      tab, slots, n, num_actions, (const uint32_t*)stats);
  HZ_LAUNCH_CHECK("k_wave_unpack");
  return HZ_OK;
}

int hz_wave_policy(void* stream, int device, const hz_policy_ticket* tickets, int count, int slots, int n,
                   int num_actions, const int32_t* stats) {
  const char* fn = "hz_wave_policy";
  if (!tickets) { set_error("%s: NULL ticket table", fn); return HZ_ERR_ARG; }
  if (slots < 1 || slots > kWaveMaxSlots) { set_error("%s: slots = %d, must be 1..%d", fn, slots, kWaveMaxSlots); return HZ_ERR_ARG; }
  if (count < 1 || count > slots) { set_error("%s: count = %d, must be 1..slots (%d)", fn, count, slots); return HZ_ERR_ARG; }
  if (n < 1 || (int64_t)slots * n > kWaveMaxRows) {
    set_error("%s: n = %d, must be >= 1 with slots * n <= %lld", fn, n, (long long)kWaveMaxRows);
    return HZ_ERR_ARG;
  }
  if (num_actions < 1 || num_actions > 32) { set_error("%s: num_actions = %d, must be 1..32", fn, num_actions); return HZ_ERR_ARG; }
  if (!stats) { set_error("%s: NULL statistics buffer", fn); return HZ_ERR_ARG; }
  for (int k = 0; k < count; ++k) {
    if (!tickets[k].out) { set_error("%s: ticket %d has a NULL output", fn, k); return HZ_ERR_ARG; }
  }
  DeviceGuard dg(device);
  if (!dg.ok) return fail_cuda(cudaGetLastError(), fn);
  if (int rc = check_ptr(fn, "statistics buffer", stats, device, 4)) return rc;
  for (int k = 0; k < count; ++k) {
    if (int rc = check_ptr(fn, "ticket mask", tickets[k].mask, device, 1)) return rc;
    if (int rc = check_ptr(fn, "ticket out", tickets[k].out, device, 8)) return rc;
  }
  PolicyTable tab{};
  for (int k = 0; k < count; ++k) tab.t[k] = tickets[k];
  k_wave_policy<<<dim3((n + kPolicyThreads - 1) / kPolicyThreads, count), kPolicyThreads, 0, (cudaStream_t)stream>>>(
      tab, n, num_actions, stats);
  HZ_LAUNCH_CHECK("k_wave_policy");
  return HZ_OK;
}

#pragma GCC visibility pop
}  // extern "C"
