// "Next" rows of the scope table (SURVEY.md §8f N3, N4): what the self-play actor does with a search
// result besides acting on it.
//   hz_traj_begin / hz_traj_append / hz_traj_pack
//       GameHistory.init / store_search_stats / append (/root/reference/core/game.py:73-93,143-148,
//       189-204) for N games at once: per game a record of (observation, action, reward, root child
//       visit counts, root value, legal mask) per move kept in HBM, closed when the game reports done
//       and handed to the host episode by episode in the replay layout (game.py:136-140, `save_file`).
//       `banks` >= 2 banks per game, used round-robin: finished episodes wait in their banks for
//       hz_traj_pack while the next episode of that game is recorded into the next free one.
//   hz_traj_record_u8
//       hz_traj_append + hz_traj_begin(mask = done) as one launch over byte rows: the recording self-play
//       engine on the frame ring (the env kernel hands over the terminal rows of finished games apart).
//   hz_visit_policy
//       visit counts -> policy targets with the out-of-trajectory mask of the reanalyze caller
//       (/root/reference/core/reanalyze_worker.py:352-367; store_search_stats, game.py:194-197).
//
// Observations of this environment are 0/1 valued, so they are recorded as bytes (exact).
#include "hz_common.cuh"

namespace hz {

constexpr int kTrajWarps = 4;

struct TrajDims {
  int64_t obs_rows, legal_rows;  // rows per bank: stack + max_len, max_len + 1
};

__device__ __forceinline__ TrajDims traj_dims(const hz_traj_view& v) {
  return TrajDims{(int64_t)v.stack + v.max_len, (int64_t)v.max_len + 1};
}

// float 0/1 row -> bytes, `copies` consecutive destination rows
__device__ __forceinline__ void put_obs(uint8_t* dst, const float* src, int dim, int copies, int lane) {
  for (int j = lane; j < dim; j += HZ_WARP) {
    const uint8_t b = src[j] != 0.0f ? 1 : 0;
    for (int c = 0; c < copies; ++c) dst[(size_t)c * dim + j] = b;
  }
}

__global__ void __launch_bounds__(kTrajWarps* HZ_WARP)
    k_traj_begin(hz_traj_view v, const float* __restrict__ obs, int64_t ld_obs, const float* __restrict__ legal,
                 const uint8_t* __restrict__ mask) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * kTrajWarps + (threadIdx.x >> 5);
  if (i >= v.num || (mask && !mask[i])) return;
  const TrajDims d = traj_dims(v);
  const int b = v.bank[i];
  if (v.finished[(size_t)v.banks * i + b]) {   // every bank holds an unflushed episode: the host did not pack in time
    if (lane == 0) atomicCAS(v.overflow, 0, i + 1);
    return;
  }
  const size_t gb = (size_t)v.banks * i + b;
  put_obs(v.obs + gb * d.obs_rows * v.obs_dim, obs + (size_t)i * ld_obs, v.obs_dim, v.stack, lane);
  if (lane < v.actions) v.legal[gb * d.legal_rows * v.actions + lane] = legal[(size_t)i * v.actions + lane] != 0.0f;
  if (lane == 0) v.len[gb] = 0;
}

__global__ void __launch_bounds__(kTrajWarps* HZ_WARP)
    k_traj_append(hz_traj_view v, const int32_t* __restrict__ actions, const float* __restrict__ obs, int64_t ld_obs,
                  const float* __restrict__ legal, const int32_t* __restrict__ reward,
                  const int32_t* __restrict__ visits, const float* __restrict__ root_values,
                  const uint8_t* __restrict__ done, const uint8_t* __restrict__ active) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * kTrajWarps + (threadIdx.x >> 5);
  if (i >= v.num || (active && !active[i])) return;
  const TrajDims d = traj_dims(v);
  const int b = v.bank[i];
  const size_t gb = (size_t)v.banks * i + b;
  const int t = v.len[gb];
  if (t >= v.max_len || v.finished[gb]) {
    if (lane == 0) atomicCAS(v.overflow, 0, i + 1);
    return;
  }
  // store_search_stats (game.py:189-204): the raw counts are kept; the division by their sum is done
  // in double precision when the episode is handed over, as Python's visit_count / sum_visits
  if (lane < v.actions) {
    v.visits[(gb * v.max_len + t) * v.actions + lane] = visits[(size_t)i * v.actions + lane];
    v.legal[(gb * d.legal_rows + t + 1) * v.actions + lane] = legal[(size_t)i * v.actions + lane] != 0.0f;
  }
  __syncwarp();   // every lane has read len / bank / finished before lane 0 updates them
  // append (game.py:143-148)
  put_obs(v.obs + (gb * d.obs_rows + v.stack + t) * v.obs_dim, obs + (size_t)i * ld_obs, v.obs_dim, 1, lane);
  if (lane == 0) {
    v.action[gb * v.max_len + t] = actions[i];
    v.reward[gb * v.max_len + t] = reward[i];
    v.root_value[gb * v.max_len + t] = root_values[i];
    v.len[gb] = t + 1;
    if (done && done[i]) {   // game_over (game.py:176-187): the episode is complete; record on in the next bank
      v.finished[gb] = 1;
      v.bank[i] = (uint8_t)((b + 1) % v.banks);
    }
  }
}

// byte 0/1 row -> bytes, `copies` consecutive destination rows (any non-zero byte is recorded as 1, as put_obs does)
__device__ __forceinline__ void put_obs_u8(uint8_t* dst, const uint8_t* src, int dim, int copies, int lane) {
  for (int j = lane; j < dim; j += HZ_WARP) {
    const uint8_t b = src[j] != 0 ? 1 : 0;
    for (int c = 0; c < copies; ++c) dst[(size_t)c * dim + j] = b;
  }
}

// k_traj_append followed by k_traj_begin(mask = done) in one launch, from byte rows: a finished game appends its
// terminal row (term_*) and begins the next episode from next_*; every other game appends next_*
__global__ void __launch_bounds__(kTrajWarps* HZ_WARP)
    k_traj_record_u8(hz_traj_view v, const int32_t* __restrict__ actions, const int32_t* __restrict__ reward,
                     const int32_t* __restrict__ visits, const float* __restrict__ root_values,
                     const uint8_t* __restrict__ done, const uint8_t* __restrict__ next_obs, int64_t ld_next,
                     const uint8_t* __restrict__ next_legal, const uint8_t* __restrict__ term_obs, int64_t ld_term,
                     const uint8_t* __restrict__ term_legal, const uint8_t* __restrict__ active) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * kTrajWarps + (threadIdx.x >> 5);
  if (i >= v.num) return;
  const TrajDims d = traj_dims(v);
  const bool fin = done[i] != 0;
  int b = v.bank[i];
  if (!active || active[i]) {
    const size_t gb = (size_t)v.banks * i + b;
    const int t = v.len[gb];
    if (t >= v.max_len || v.finished[gb]) {
      if (lane == 0) atomicCAS(v.overflow, 0, i + 1);
    } else {
      const uint8_t* obs = fin ? term_obs + (size_t)i * ld_term : next_obs + (size_t)i * ld_next;
      const uint8_t* legal = (fin ? term_legal : next_legal) + (size_t)i * v.actions;
      if (lane < v.actions) {
        v.visits[(gb * v.max_len + t) * v.actions + lane] = visits[(size_t)i * v.actions + lane];
        v.legal[(gb * d.legal_rows + t + 1) * v.actions + lane] = legal[lane] != 0;
      }
      put_obs_u8(v.obs + (gb * d.obs_rows + v.stack + t) * v.obs_dim, obs, v.obs_dim, 1, lane);
      __syncwarp();   // every lane has read len / bank / finished before lane 0 updates them
      if (lane == 0) {
        v.action[gb * v.max_len + t] = actions[i];
        v.reward[gb * v.max_len + t] = reward[i];
        v.root_value[gb * v.max_len + t] = root_values[i];
        v.len[gb] = t + 1;
        if (fin) {
          v.finished[gb] = 1;
          v.bank[i] = (uint8_t)((b + 1) % v.banks);
        }
      }
      if (fin) b = (b + 1) % v.banks;
    }
  }
  if (!fin) return;
  // begin: the bank just moved to is one this launch has not written (banks >= 2), so every lane may read its flag
  const size_t gb = (size_t)v.banks * i + b;
  if (v.finished[gb]) {
    if (lane == 0) atomicCAS(v.overflow, 0, i + 1);
    return;
  }
  put_obs_u8(v.obs + gb * d.obs_rows * v.obs_dim, next_obs + (size_t)i * ld_next, v.obs_dim, v.stack, lane);
  if (lane < v.actions) v.legal[gb * d.legal_rows * v.actions + lane] = next_legal[(size_t)i * v.actions + lane] != 0;
  __syncwarp();   // every lane has read len before lane 0 rewrites it (append overflow with the bank unchanged)
  if (lane == 0) v.len[gb] = 0;
}

// one CTA per finished episode: copy its rows into the packed staging buffers and free the bank
__global__ void __launch_bounds__(256)
    k_traj_pack(hz_traj_view v, const int32_t* __restrict__ ep_game, const int32_t* __restrict__ ep_bank,
                const int64_t* __restrict__ step_off, uint8_t* __restrict__ out_obs, uint8_t* __restrict__ out_legal,
                int32_t* __restrict__ out_action, int32_t* __restrict__ out_reward, int32_t* __restrict__ out_visits,
                float* __restrict__ out_root) {
  const int e = blockIdx.x;
  const TrajDims d = traj_dims(v);
  const size_t gb = (size_t)v.banks * ep_game[e] + ep_bank[e];
  const int64_t T = v.len[gb], s0 = step_off[e];
  // episode e owns obs rows [s0 + e*stack, ...), legal rows [s0 + e, ...), step rows [s0, s0 + T)
  const uint8_t* so = v.obs + gb * d.obs_rows * v.obs_dim;
  uint8_t* po = out_obs + (s0 + (int64_t)e * v.stack) * v.obs_dim;
  const int64_t nb = (v.stack + T) * v.obs_dim;
  if ((((uintptr_t)so | (uintptr_t)po) & 15) == 0) {
    for (int64_t k = threadIdx.x; k < (nb >> 4); k += blockDim.x)
      reinterpret_cast<uint4*>(po)[k] = reinterpret_cast<const uint4*>(so)[k];
    for (int64_t k = (nb & ~(int64_t)15) + threadIdx.x; k < nb; k += blockDim.x) po[k] = so[k];
  } else {
    for (int64_t k = threadIdx.x; k < nb; k += blockDim.x) po[k] = so[k];
  }
  const uint8_t* sl = v.legal + gb * d.legal_rows * v.actions;
  uint8_t* pl = out_legal + (s0 + e) * v.actions;
  for (int64_t k = threadIdx.x; k < (T + 1) * v.actions; k += blockDim.x) pl[k] = sl[k];
  const int32_t* sv = v.visits + gb * v.max_len * v.actions;
  for (int64_t k = threadIdx.x; k < T * v.actions; k += blockDim.x) out_visits[s0 * v.actions + k] = sv[k];
  for (int64_t k = threadIdx.x; k < T; k += blockDim.x) {
    out_action[s0 + k] = v.action[gb * v.max_len + k];
    out_reward[s0 + k] = v.reward[gb * v.max_len + k];
    out_root[s0 + k] = v.root_value[gb * v.max_len + k];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    v.finished[gb] = 0;
    v.len[gb] = 0;
  }
}

__global__ void k_visit_policy(const int32_t* __restrict__ visits, const uint8_t* __restrict__ mask, int num, int A,
                               double* __restrict__ out64, float* __restrict__ out32) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num) return;
  visit_policy_row(visits + (size_t)i * A, !mask || mask[i], A, out64 ? out64 + (size_t)i * A : nullptr,
                   out32 ? out32 + (size_t)i * A : nullptr);
}

static int check_view(const hz_traj_view* v, const char* who) {
  if (!v || !v->obs || !v->legal || !v->action || !v->reward || !v->visits || !v->root_value || !v->len || !v->bank ||
      !v->finished || !v->overflow || v->num <= 0 || v->obs_dim <= 0 || v->actions <= 0 || v->actions > 32 ||
      v->stack <= 0 || v->max_len <= 0 || v->banks < 2 || v->banks > 255) {
    set_error("%s: malformed hz_traj_view", who);
    return HZ_ERR_ARG;
  }
  return HZ_OK;
}

}  // namespace hz

using namespace hz;

extern "C" {
#pragma GCC visibility push(default)

int hz_traj_begin(void* stream, const hz_traj_view* v, const float* obs, int64_t ld_obs, const float* legal,
                  const uint8_t* mask) {
  if (int rc = check_view(v, "hz_traj_begin")) return rc;
  if (!obs || !legal || ld_obs < v->obs_dim) { set_error("hz_traj_begin: bad observation argument"); return HZ_ERR_ARG; }
  k_traj_begin<<<(v->num + kTrajWarps - 1) / kTrajWarps, kTrajWarps * HZ_WARP, 0, (cudaStream_t)stream>>>(
      *v, obs, ld_obs, legal, mask);
  HZ_LAUNCH_CHECK("k_traj_begin");
  return HZ_OK;
}

int hz_traj_append(void* stream, const hz_traj_view* v, const int32_t* actions, const float* obs, int64_t ld_obs,
                   const float* legal, const int32_t* reward, const int32_t* visits, const float* root_values,
                   const uint8_t* done, const uint8_t* active) {
  if (int rc = check_view(v, "hz_traj_append")) return rc;
  if (!actions || !obs || !legal || !reward || !visits || !root_values || ld_obs < v->obs_dim) {
    set_error("hz_traj_append: NULL argument or row stride smaller than the observation");
    return HZ_ERR_ARG;
  }
  k_traj_append<<<(v->num + kTrajWarps - 1) / kTrajWarps, kTrajWarps * HZ_WARP, 0, (cudaStream_t)stream>>>(
      *v, actions, obs, ld_obs, legal, reward, visits, root_values, done, active);
  HZ_LAUNCH_CHECK("k_traj_append");
  return HZ_OK;
}

int hz_traj_record_u8(void* stream, const hz_traj_view* v, const int32_t* actions, const int32_t* reward,
                      const int32_t* visits, const float* root_values, const uint8_t* done, const uint8_t* next_obs,
                      int64_t ld_next, const uint8_t* next_legal, const uint8_t* term_obs, int64_t ld_term,
                      const uint8_t* term_legal, const uint8_t* active) {
  if (int rc = check_view(v, "hz_traj_record_u8")) return rc;
  if (!actions || !reward || !visits || !root_values || !done || !next_obs || !next_legal || !term_obs || !term_legal ||
      ld_next < v->obs_dim || ld_term < v->obs_dim) {
    set_error("hz_traj_record_u8: NULL argument or row stride smaller than the observation");
    return HZ_ERR_ARG;
  }
  k_traj_record_u8<<<(v->num + kTrajWarps - 1) / kTrajWarps, kTrajWarps * HZ_WARP, 0, (cudaStream_t)stream>>>(
      *v, actions, reward, visits, root_values, done, next_obs, ld_next, next_legal, term_obs, ld_term, term_legal, active);
  HZ_LAUNCH_CHECK("k_traj_record_u8");
  return HZ_OK;
}

int hz_traj_pack(void* stream, const hz_traj_view* v, int num_episodes, const int32_t* ep_game, const int32_t* ep_bank,
                 const int64_t* step_off, uint8_t* out_obs, uint8_t* out_legal, int32_t* out_action,
                 int32_t* out_reward, int32_t* out_visits, float* out_root) {
  if (int rc = check_view(v, "hz_traj_pack")) return rc;
  if (num_episodes == 0) return HZ_OK;
  if (num_episodes < 0 || !ep_game || !ep_bank || !step_off || !out_obs || !out_legal || !out_action || !out_reward ||
      !out_visits || !out_root) {
    set_error("hz_traj_pack: bad argument");
    return HZ_ERR_ARG;
  }
  k_traj_pack<<<num_episodes, 256, 0, (cudaStream_t)stream>>>(*v, ep_game, ep_bank, step_off, out_obs, out_legal,
                                                              out_action, out_reward, out_visits, out_root);
  HZ_LAUNCH_CHECK("k_traj_pack");
  return HZ_OK;
}

int hz_visit_policy(void* stream, const int32_t* visits, const uint8_t* mask, int num, int num_actions, double* out64,
                    float* out32) {
  if (!visits || num <= 0 || num_actions <= 0 || (!out64 && !out32)) {
    set_error("hz_visit_policy: bad argument");
    return HZ_ERR_ARG;
  }
  k_visit_policy<<<(num + 127) / 128, 128, 0, (cudaStream_t)stream>>>(visits, mask, num, num_actions, out64, out32);
  HZ_LAUNCH_CHECK("k_visit_policy");
  return HZ_OK;
}

#pragma GCC visibility pop
}  // extern "C"
