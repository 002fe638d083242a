/* hzb200 — C ABI of the B200-native HanabiZero self-play hot path.
 *
 * One shared library (hanabizero_b200/csrc/libhzb200.so, sm_100a) replaces the two native
 * libraries the reference binds on this path:
 *   (1) the Cython extension `core.ctree.cytree` over core/ctree/{cnode,cminimax}.{h,cpp}
 *       (/root/reference/core/ctree/cytree.pyx:17-101, ctree.pxd:9-77), and
 *   (2) `libpyhanabi.so`, the cffi-loaded C API over envs/hanabi/hanabi_lib
 *       (/root/reference/envs/hanabi/pyhanabi.h:24-195), as driven by HanabiEnv.reset/step
 *       (/root/reference/envs/hanabi/rl_env.py:148-267, 292-442).
 *
 * Conventions: every function returns 0 on success and a negative hz_status on failure
 * (hz_last_error() then holds a message, thread-local).  All `dev` pointers are device memory on
 * the handle's device; `stream` is a cudaStream_t passed as void*.  No call synchronises the
 * stream or allocates unless stated ("sync").  Batches are structure-of-arrays over trees/games;
 * tree i / game i of a batch is the reference's roots[i] / envs[i].
 */
#ifndef HZB200_H
#define HZB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hz_trees hz_trees;
typedef struct hz_envs hz_envs;

typedef enum {
  HZ_OK = 0,
  HZ_ERR_ARG = -1,      /* bad argument (NULL handle, size mismatch, x out of capacity ...) */
  HZ_ERR_CUDA = -2,     /* a CUDA runtime call or launch failed */
  HZ_ERR_STATE = -3,    /* call order violated (backprop without traverse, step before reset ...) */
  HZ_ERR_ILLEGAL = -4   /* an illegal Hanabi move was submitted (reference: REQUIRE -> abort,
                           hanabi_state.cc:222) */
} hz_status;

const char* hz_last_error(void);
int hz_version(void);
/* number of kernels this library has launched in this process (bench.py "gpu_launches") */
int64_t hz_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Tree batch.  Replaces cytree.Roots + the per-tree node pools (CRoots, cnode.h:43-60;
 * Roots.__cinit__, cytree.pyx:42-45) and the search paths held by ResultsWrapper/CSearchResults
 * (cnode.h:62-73).  Capacity: `max_sims` expansions per tree beyond the root.
 * ------------------------------------------------------------------------------------------ */
int hz_trees_create(hz_trees** out, int device, int num_trees, int num_actions, int max_sims); /* sync */
int hz_trees_destroy(hz_trees* t);                                                             /* sync */
int hz_trees_num(const hz_trees* t);
int hz_trees_actions(const hz_trees* t);
int hz_trees_capacity(const hz_trees* t);

/* CRoots::prepare / prepare_no_noise (cnode.cpp:247-259; cytree.pyx:47-51): masked softmax
 * expansion of every root with hidden index (0, i), then the Dirichlet-noise mix.
 * noises == NULL selects prepare_no_noise.  All inputs dev: noises/logits float[N][A],
 * rewards float[N], masks int32[N][A] (0 = illegal).  Also discards any previous search. */
int hz_trees_prepare(hz_trees* t, void* stream, float exploration_fraction, const float* noises,
                     const float* rewards, const float* logits, const int32_t* masks);

/* cmulti_traverse (cnode.cpp:407-441; cytree.multi_traverse, cytree.pyx:97-101) with the tie
 * rule rand()==0.  minmax: dev float[N][2] = {minimum, maximum} per tree — the storage of
 * CMinMaxStatsList (cminimax.h:13-36), owned by the caller like the reference's separate
 * MinMaxStatsList object; value_delta_max is CMinMaxStats::value_delta_max.
 * Outputs (dev, any may be NULL): out_ix/out_iy int32[N] = the leaf's PARENT hidden-state
 * index, out_action int32[N] = last action, out_action64 int64[N] (same, for torch .long()).
 * If pool != NULL, also gathers the parent hidden state rows (mcts.py:31-35 done on device):
 *   out_hidden[i, :] = pool[(ix*N + iy) * row_bytes ...], row_bytes % 16 == 0. */
int hz_trees_traverse(hz_trees* t, void* stream, int pb_c_base, float pb_c_init, float discount,
                      const float* minmax, float value_delta_max, int32_t* out_ix, int32_t* out_iy,
                      int32_t* out_action, int64_t* out_action64, const void* pool,
                      void* out_hidden, int row_bytes);

/* cmulti_back_propagate (cnode.cpp:337-344; cytree.multi_back_propagate, cytree.pyx:87-94):
 * expand every leaf found by the last traverse with hidden index (hidden_state_index_x, i) and
 * all-legal softmax priors, back-propagate `values` along the path, then refresh the per-tree
 * min/max over all expanded non-root nodes (cback_propagate + update_tree_q, cnode.cpp:296-335).
 * rewards/values float[N], logits float[N][A] (dev).  sanitize_nan != 0 zeroes NaN logits first
 * (what core/mcts.py:48-49 does on the host).  minmax is written. */
int hz_trees_backprop(hz_trees* t, void* stream, int hidden_state_index_x, float discount,
                      const float* rewards, const float* values, const float* logits,
                      int sanitize_nan, float* minmax);

/* Fused step for the device-resident search loop: backprop of simulation k immediately followed
 * by the traverse (+ gather) of simulation k+1 in ONE launch.  Same results as calling
 * hz_trees_backprop then hz_trees_traverse. */
int hz_trees_backprop_traverse(hz_trees* t, void* stream, int hidden_state_index_x, float discount,
                               const float* rewards, const float* values, const float* logits,
                               int sanitize_nan, float* minmax, float value_delta_max,
                               int pb_c_base, float pb_c_init, int32_t* out_ix, int32_t* out_iy,
                               int32_t* out_action, int64_t* out_action64, const void* pool,
                               void* out_hidden, int row_bytes);

/* One launch per simulation for the device-resident loop, consuming the network's RAW outputs:
 *   x == 0 : traverse only (first simulation after prepare);
 *   x >= 1 : decode value/reward of simulation x from their categorical logits
 *            (core/config.py:210-232), expand + back-propagate (as hz_trees_backprop), store the new
 *            node's hidden state into pool[x], then (do_traverse != 0) traverse for simulation
 *            x+1 and write the next network input batch: the parent's hidden state followed by
 *            one-hot(last action) (the concat of dynamics(), config/hanabi_control/model.py:199-203). */
typedef struct hz_search_io {
  /* network outputs of simulation x, row-major, `elem_bytes` per element (2 = half, 4 = float) */
  const void* value_logits;   int64_t ld_value;    /* [N][support_width] */
  const void* reward_logits;  int64_t ld_reward;   /* [N][support_width] */
  const void* policy_logits;  int64_t ld_policy;   /* [N][A] */
  const void* next_state;     int64_t ld_state;    /* [N][state_cols], or NULL when the network wrote the new
                                                    * hidden state straight into pool[x] (no copy in the kernel) */
  const float* support;       /* dev float[support_width] */
  int32_t support_width;      /* <= 256 */
  float support_delta;
  int32_t elem_bytes;
  int32_t sanitize_nan;       /* zero NaN policy logits (core/mcts.py:48-49) */
  /* hidden-state pool and the batch handed to the network */
  void* pool;                 /* [capacity+1][N][state_cols], elem_bytes each */
  int32_t state_cols;         /* state_cols * elem_bytes must be a multiple of 16 */
  void* out_batch;            /* [N][ld_batch]: state_cols of hidden state, then onehot_cols of one-hot */
  int64_t ld_batch;           /* elements; ld_batch * elem_bytes multiple of 16 */
  int32_t onehot_cols;        /* 0 (no one-hot columns are written) or num_actions..32; columns >= num_actions are
                               * written as zero.  1..num_actions-1 is an argument error: an action without a column
                               * would reach the network as an all-zero one-hot */
  int32_t* out_ix;            /* optional int32[N]: parent hidden-state index x */
  int32_t* out_action;        /* optional int32[N]: last action */
  /* search constants */
  float* minmax;              /* dev float[N][2], read and written */
  float value_delta_max;
  float discount;
  int32_t pb_c_base;
  float pb_c_init;
  /* != 0: launch with programmatic stream serialization — the kernel fetches its tree state while the preceding
   * kernel of the stream drains and synchronises on it before reading the network outputs.  The caller guarantees
   * that the preceding kernel is not the previous tree step (there is at least one network kernel in between). */
  int32_t programmatic_launch;
  /* > 0: stage at most this many expanded nodes' records in shared memory (and none of q).  0 = as much of the tree as
   * fits, the fastest choice for a search that runs alone.  With several searches in flight on different streams a
   * small limit (4) is better: the launch then needs ~6 KB of shared memory per CTA and shares SMs with the library
   * GEMM CTAs of the other searches instead of waiting for SMs without one. */
  int32_t stage_limit;
} hz_search_io;
int hz_trees_search_step(hz_trees* t, void* stream, int x, int do_traverse, const hz_search_io* io);

/* After replaying a CUDA graph that contains the calls above, the handle's host-side progress
 * (number of completed back-propagations since prepare) must be restored by hand: a replay runs
 * the kernels but not the host code.  expansions in [0, capacity]. */
int hz_trees_set_progress(hz_trees* t, int expansions);

/* Tie rule of cselect_child (cnode.cpp:346-374).  The reference draws rand() % ties over the children whose score is
 * within 1e-6 of the best (after srand(gettimeofday) per traverse, cnode.cpp:409-411).  mode 0 (default, the parity
 * contract with the rand() == 0 build of the reference): the first element of that list.  mode 1: a uniform draw
 * from a counter-based generator keyed by (seed, tree_offset + tree index, simulations completed, depth) — the same
 * tie LIST as the reference, a reproducible draw instead of the clock-seeded libc stream.  tree_offset is the global
 * index of this batch's tree 0, so a root batch sharded over ranks draws exactly what the unsharded batch draws.
 * Takes effect at the next hz_trees_prepare (which stores the rule in device memory, so a captured CUDA graph of the
 * simulation loop follows the rule of the search it is replayed for); pass a fresh seed per search. */
int hz_trees_set_tie_break(hz_trees* t, int mode, uint64_t seed, int tree_offset);

/* CRoots::get_distributions / get_values (cnode.cpp:276-292): out_visits int32[N][A] (dev),
 * out_values float[N] (dev). */
int hz_trees_root_stats(hz_trees* t, void* stream, int32_t* out_visits, float* out_values);

/* CRoots::get_trajectories (cnode.cpp:266-274): out int32[N][max_len] (dev), -1 padded. */
int hz_trees_trajectories(hz_trees* t, void* stream, int32_t* out, int max_len);

/* Test/inspection export: per tree and expansion index x in [1, cap]: reward, value_sum (dev
 * float[N][cap]) and visit_count (dev int32[N][cap]); entries past the last expansion are 0.
 * out_path_len int32[N] = length of the last search path (nodes incl. root). NULLs allowed. */
int hz_trees_export(hz_trees* t, void* stream, int cap, float* out_reward, float* out_value_sum,
                    int32_t* out_visits, float* out_root_priors, int32_t* out_path_len);

/* mcts.py:31-35 as a standalone op: out[i,:] = pool[(ix[i]*num + iy[i]) * row_bytes ...]. */
int hz_gather_hidden(void* stream, const void* pool, const int32_t* ix, const int32_t* iy,
                     void* out, int num, int row_bytes);

/* ------------------------------------------------------------------------------------------
 * Hanabi game batch.  Replaces, per game i, one HanabiGame + HanabiState + ObservationEncoder
 * (pyhanabi.h: NewGame, NewState, StateApplyMove, StateDealRandomCard, NewObservation,
 * EncodeObservation, EncodeOwnHandObservation, ObsGetLegalMove, StateScore,
 * StateEndOfGameStatus) as sequenced by HanabiEnv.reset/step.
 * preset: 0 = "Hanabi-Full", 1 = "Hanabi-Small" (rl_env.py:110-131).  seeds: HOST int32[N],
 * game i seeds its own std::mt19937 with seeds[i] (hanabi_game.cc:43-51); the stream persists
 * across resets like the reference's game object.
 * ------------------------------------------------------------------------------------------ */
int hz_envs_create(hz_envs** out, int device, int num_games, int preset, const int32_t* seeds); /* sync */
int hz_envs_destroy(hz_envs* e);                                                                /* sync */
/* dims: [enc_len, own_len, players, actions, colors, ranks, hand_size, max_info, max_life,
 *        local_dim, global_dim, state_dump_len] */
int hz_envs_dims(const hz_envs* e, int32_t* out12);

/* HanabiEnv.reset (rl_env.py:148-267) for the games with reset_mask[i] != 0 (dev uint8[N];
 * NULL = all games). Observations are produced by hz_envs_observe. */
int hz_envs_reset(hz_envs* e, void* stream, const uint8_t* reset_mask);

/* HanabiEnv.step (rl_env.py:292-442) for every game with active[i] != 0 (dev uint8[N]; NULL =
 * all): apply move uid actions[i] (dev int32[N]), deal while chance, then reward = score delta,
 * done, score.  out_reward/out_score int32[N], out_done uint8[N] (dev).  An illegal action
 * leaves that game untouched and raises the sticky error flag read by hz_envs_check. */
int hz_envs_step(hz_envs* e, void* stream, const int32_t* actions, const uint8_t* active,
                 int32_t* out_reward, uint8_t* out_done, int32_t* out_score);

/* The observation tuple HanabiEnv returns for the current player (rl_env.py:254-263, 426-434):
 * out_global float[N][global_dim] = own-hand ‖ canonical encoding ‖ turn one-hot,
 * out_local float[N][local_dim], out_legal float[N][actions] (dev; any may be NULL).
 * ld_global/ld_local = row stride in elements (>= dim; lets the caller write straight into a
 * frame-stack buffer). */
int hz_envs_observe(hz_envs* e, void* stream, float* out_global, int64_t ld_global,
                    float* out_local, int64_t ld_local, float* out_legal);

/* step + auto-reset of finished games + observe in one launch (the self-play inner loop). */
int hz_envs_step_observe(hz_envs* e, void* stream, const int32_t* actions, const uint8_t* active,
                         int auto_reset, int32_t* out_reward, uint8_t* out_done, int32_t* out_score,
                         float* out_global, int64_t ld_global, float* out_local, int64_t ld_local,
                         float* out_legal);

/* The same two calls with byte-valued outputs: every element is 0 or 1 as uint8 — the value type
 * the reference encoder itself emits (std::vector<int> of 0/1, canonical_encoders.cc:441-486,
 * serialised by pyhanabi.cc:855-895) at a quarter of the float32 traffic.  Row strides in bytes. */
int hz_envs_observe_u8(hz_envs* e, void* stream, uint8_t* out_global, int64_t ld_global, uint8_t* out_local,
                       int64_t ld_local, uint8_t* out_legal);
int hz_envs_step_observe_u8(hz_envs* e, void* stream, const int32_t* actions, const uint8_t* active,
                            int auto_reset, int32_t* out_reward, uint8_t* out_done, int32_t* out_score,
                            uint8_t* out_global, int64_t ld_global, uint8_t* out_local, int64_t ld_local,
                            uint8_t* out_legal);
/* hz_envs_step_observe_u8 with auto-reset, for a caller that records trajectories: a finished game's TERMINAL
 * observation (what auto_reset = 0 would have written, the row GameHistory.append takes, rl_env.py:426-434) goes to
 * out_term (uint8[N][ld_term]) and its legal mask to out_term_legal (uint8[N][actions]; non-zero at terminal states:
 * the reference has no terminal check), then the game is re-dealt and the first observation of its next episode goes
 * to the usual output row.  Rows of games that did not finish are left as they were.  Exactly one of out_global /
 * out_local is given, and the terminal rows are in that view (ld_term >= its width); out_term / out_term_legal may be
 * NULL like the other outputs. */
int hz_envs_step_observe_u8_terminal(hz_envs* e, void* stream, const int32_t* actions, const uint8_t* active,
                                     int32_t* out_reward, uint8_t* out_done, int32_t* out_score, uint8_t* out_global,
                                     int64_t ld_global, uint8_t* out_local, int64_t ld_local, uint8_t* out_legal,
                                     uint8_t* out_term, int64_t ld_term, uint8_t* out_term_legal);

/* The host-facing form of the same launch: ONE bit-packed row of uint32 words per game (dev, row stride ld_words >=
 * W + 4 with W = ceil(global_dim / 32): 25 for Hanabi-Full, 7 for Hanabi-Small):
 *   words [0, W)   the global observation, bit j = (row[j >> 5] >> (j & 31)) & 1 — the encoder emits 0/1 values
 *                  (canonical_encoders.cc:441-486), so 785 of them are 100 bytes, not 785 or 3140; the local
 *                  observation is bits [own_len, global_dim) of the same string (rl_env.py:261-262)
 *   word  W        legal-move mask, bit a = move uid a is legal (rl_env.py:263)
 *   words W+1..3   reward (int32), done (0/1), score of the step (rl_env.py:436-442)
 * actions == NULL observes without stepping (reward 0).  A host caller copies N * (W + 4) * 4 bytes per step.
 * out_meta (optional, dev uint32[N][4], 16-byte aligned): the four trailing words {legal mask, reward, done, score} go
 * there instead (rows then need only W words) — a host policy that looks at the legal mask reads 16 contiguous bytes
 * per game instead of one word out of every 116-byte row. */
int hz_envs_step_observe_bits(hz_envs* e, void* stream, const int32_t* actions, const uint8_t* active, int auto_reset,
                              uint32_t* out_bits, int64_t ld_words, uint32_t* out_meta);
/* Host-facing step for callers that keep actions and results in page-locked HOST memory (a vectorised stand-in for
 * the per-step pyhanabi.h calls of HanabiEnv.step, rl_env.py:292-442): h_actions (int32[N], NULL = observe only),
 * h_bits / h_meta as in hz_envs_step_observe_bits but HOST pointers.  No staging copies: pinned memory is
 * device-addressable, the kernel reads and writes it directly, so a step is one launch + one event record on
 * `stream`.  hz_envs_host_wait blocks the calling thread until the last hz_envs_host_step of this handle has landed in
 * host memory.  Neither call holds any lock: one host thread per game batch may drive its own handle. */
int hz_envs_host_step(hz_envs* e, void* stream, const int32_t* h_actions, int auto_reset, uint32_t* h_bits,
                      int64_t ld_words, uint32_t* h_meta);
int hz_envs_host_wait(hz_envs* e);
/* Fused random policy for device-resident random play (rollouts, env throughput runs): after this call every
 * observing launch of the handle (hz_envs_observe*, hz_envs_step_observe*, hz_envs_host_step) also writes, for every
 * game it observes, a uniformly random legal move of the observed position into next_actions (dev int32[N], caller
 * owned; 0 for a finished game) — pass the same buffer as `actions` of the next step and a whole random-play step is
 * ONE launch.  Draw d of game i is the k-th legal move with k from the generator of hz_host_random_legal keyed
 * (seed, i, step = d): the host twin reproduces any pick.  The per-game draw counters live on the device (CUDA-graph
 * replays keep advancing them) and are reset to 0 by this call; next_actions == NULL switches the policy off. */
int hz_envs_set_random_policy(hz_envs* e, void* stream, int32_t* next_actions, uint64_t seed);
/* HOST helper for callers that drive the games from the CPU through the packed rows (no device work): a uniformly
 * random legal move per game from word `legal_word` (= W) of each host row, counter-based (seed, game, step). */
int hz_host_random_legal(const uint32_t* rows, int64_t ld_words, int legal_word, int num_games, int num_actions,
                         uint64_t seed, uint32_t step, int32_t* out_actions);

/* sync: returns HZ_ERR_ILLEGAL if any game saw an illegal action since the last check
 * (out_game = first offending game index), clearing the flag. */
int hz_envs_check(hz_envs* e, void* stream, int32_t* out_game);

/* Full hidden state of every game for parity tests, int32[N][state_dump_len] (dev), layout of
 * oracle/hanabi_oracle.c:ohanabi_dump. */
int hz_envs_dump(hz_envs* e, void* stream, int32_t* out);

/* ------------------------------------------------------------------------------------------
 * Glue around the PyTorch network (the GEMMs stay cuBLAS): keeps value/reward decoding and the
 * layer epilogues on the device in one launch each.
 * ------------------------------------------------------------------------------------------ */
/* inverse_scalar_transform (/root/reference/core/config.py:210-232): per row softmax over `width`
 * support bins (logits dev, elem_bytes 4 = float / 2 = half, row stride ld elements), expectation
 * against support[width] (dev float), / delta, inverse of h(x)=sign(x)(sqrt(|x|+1)-1)+0.001x,
 * NaN -> 0.  out: dev float[rows]. */
int hz_support_decode(void* stream, const void* logits, int elem_bytes, const float* support,
                      float* out, int rows, int width, int64_t ld, float delta);
/* ------------------------------------------------------------------------------------------
 * "Next" rows (SURVEY.md §8f): the hops between a search and the next env step.
 * ------------------------------------------------------------------------------------------ */
/* Root exploration noise (np.random.dirichlet([alpha] * A) per root, /root/reference/core/selfplay_worker.py:279,
 * reanalyze_worker.py:343-344) from counter-based streams: Philox4x32-10 keyed by `seed`, counter (block, action,
 * root_offset + root, step); Gamma(alpha) by Marsaglia-Tsang, normalised in ascending order, rounded to float32.
 * alpha must lie in [1e-300, 1e300] (NaN and inf are rejected with HZ_ERR_ARG); 1 <= A <= 32.  For alpha < 1 a row
 * whose gammas would all underflow is rescaled by its largest one, so every row is finite and sums to 1 within
 * float32 rounding.  out float[N][A] (dev).  legal_mask (optional, float[N][A]): an entry is zeroed AFTER
 * normalisation when its mask value == 0.0f (-0.0f included); any other value, 0.5 or NaN included, leaves the entry
 * as drawn — this is not noise * legal.  hz_host_dirichlet_noise is the host twin (host pointers, no device work):
 * the same arithmetic built from IEEE float64 operations only, bit-identical output — a search can be replayed on the
 * CPU (e.g. through the reference's own cytree) with exactly the noise the device drew. */
int hz_dirichlet_noise(void* stream, float* out, int num_roots, int num_actions, double alpha, uint64_t seed,
                       uint32_t step, uint32_t root_offset, const float* legal_mask);
int hz_host_dirichlet_noise(float* out, int num_roots, int num_actions, double alpha, uint64_t seed, uint32_t step,
                            uint32_t root_offset, const float* legal_mask);

/* select_action (/root/reference/core/utils.py:280-295): visits int32[N][A] (dev; counts of illegal
 * actions are zeroed in place like the reference does), legal float[N][A], temperature double[N] or
 * NULL (= 1), uniforms double[N] in [0,1) or NULL (deterministic: first arg-max).  p[a] = pow(c[a], 1 / T)
 * in double, summed in ascending order.  Sampling follows numpy.random.choice (cdf = cumsum(p)/sum,
 * searchsorted side='right') for the given uniform.  out_action int32[N], out_entropy float[N] or NULL
 * (base-2 entropy of the visit distribution).  A row whose sum of p is 0 (no visits left on a legal move) or not
 * finite (c^(1/T) overflows: a tiny or zero temperature) has no distribution: its action is -1, which the env
 * kernels reject as an illegal move, and its entropy NaN. */
int hz_select_action(void* stream, int32_t* visits, const float* legal, const double* temperature,
                     const double* uniforms, int num, int num_actions, int32_t* out_action, float* out_entropy);
/* Frame stack on the device (core/game.py:169-174): stack float[N][depth][dim] shifts left by one
 * frame and appends obs[i] (row stride ld_obs); where done[i] != 0 every slot is filled with obs[i]
 * (first frame of the next episode replicated, selfplay_worker.py:137). */
int hz_stack_push(void* stream, float* stack, const float* obs, int64_t ld_obs, const uint8_t* done, int num,
                  int stack_depth, int dim);

/* The same frame stack as a RING of 0/1 bytes: ring uint8[N][stack_depth][padded_dim] (dev; padded_dim = frame length
 * rounded up to 16).  The env kernel writes every new observation straight into the slot holding the oldest frame
 * (hz_envs_step_observe_u8 with that slot as its output row), so a move costs no memmove at all.
 * hz_ring_gather: the network input in frame order, oldest first: out[i][j * frame_stride + d] =
 *   ring[i][(head + j) % stack_depth][d] as half (elem_bytes 2) or float (4); frame_stride >= padded_dim, both
 *   multiples of 16 (the first layer's weight columns are laid out with the same stride).
 * hz_ring_refill: games with done[i] != 0 (NULL = all) get slot src_slot copied into every other slot — the first
 *   observation of a new episode fills the whole stack (core/selfplay_worker.py:137). */
int hz_ring_gather(void* stream, const uint8_t* ring, int head, void* out, int64_t ld_out, int frame_stride, int num,
                   int stack_depth, int padded_dim, int elem_bytes);
int hz_ring_refill(void* stream, uint8_t* ring, int src_slot, const uint8_t* done, int num, int stack_depth, int padded_dim);

/* Trajectory record of N self-play games in HBM (SURVEY.md §8f N3): GameHistory.init /
 * store_search_stats / append / game_over (/root/reference/core/game.py:73-93,143-148,176-204) for a
 * whole batch.  The caller owns the buffers (device memory, zero-initialised) and passes this view.
 * `banks` >= 2 banks per game (B below), used round-robin: an episode closed by done[i] waits in its bank for
 * hz_traj_pack while the game's next episodes are recorded into the following banks.  Observations are 0/1
 * valued and kept as bytes. */
typedef struct hz_traj_view {
  uint8_t* obs;        /* [N][B][stack + max_len][obs_dim]: `stack` copies of the first frame, then one per move */
  uint8_t* legal;      /* [N][B][max_len + 1][actions]: legal mask before move t (row 0 from begin) */
  int32_t* action;     /* [N][B][max_len] */
  int32_t* reward;     /* [N][B][max_len] raw env rewards (the turn-reward reshaping of
                          selfplay_worker.py:29-39 is applied when the episode is handed over) */
  int32_t* visits;     /* [N][B][max_len][actions] root child visit counts */
  float* root_value;   /* [N][B][max_len] */
  int32_t* len;        /* [N][B] moves recorded in each bank */
  uint8_t* bank;       /* [N] bank currently written */
  uint8_t* finished;   /* [N][B] 1 = complete episode awaiting hz_traj_pack */
  int32_t* overflow;   /* [1] sticky: 1 + first game that ran out of room (episode longer than max_len,
                          or every bank full because the host did not pack in time) */
  int32_t num, obs_dim, actions, stack, max_len, banks;
} hz_traj_view;
/* GameHistory.init for the games with mask[i] != 0 (dev uint8[N], NULL = all): the first observation
 * (dev float[N][ld_obs]) fills the `stack` leading frames, the first legal mask (dev float[N][actions])
 * row 0. */
int hz_traj_begin(void* stream, const hz_traj_view* v, const float* obs, int64_t ld_obs, const float* legal,
                  const uint8_t* mask);
/* One self-play move of every game with active[i] != 0 (NULL = all): store_search_stats(visits, root_value)
 * + append(action, obs, reward, legal); done[i] != 0 closes the episode (game_over) and moves on to the next bank —
 * call hz_traj_begin with mask = done afterwards, once the env has been reset.  All pointers dev. */
int hz_traj_append(void* stream, const hz_traj_view* v, const int32_t* actions, const float* obs, int64_t ld_obs,
                   const float* legal, const int32_t* reward, const int32_t* visits, const float* root_values,
                   const uint8_t* done, const uint8_t* active);
/* One launch per move for the recording engine on the byte frame ring: per game exactly hz_traj_append followed by
 * hz_traj_begin(mask = done), from uint8 rows (non-zero = 1).  The appended observation and legal row are term_obs /
 * term_legal where done[i] != 0 (hz_envs_step_observe_u8_terminal's terminal rows) and next_obs / next_legal
 * elsewhere; a finished game then begins its next bank with `stack` copies of next_obs and legal row 0 = next_legal.
 * Row strides ld_next / ld_term in bytes (>= obs_dim), legal rows [N][actions].  done is required; active as in
 * hz_traj_append (the begin of a finished game does not look at it, as hz_traj_begin does not).  All pointers dev. */
int hz_traj_record_u8(void* stream, const hz_traj_view* v, const int32_t* actions, const int32_t* reward,
                      const int32_t* visits, const float* root_values, const uint8_t* done, const uint8_t* next_obs,
                      int64_t ld_next, const uint8_t* next_legal, const uint8_t* term_obs, int64_t ld_term,
                      const uint8_t* term_legal, const uint8_t* active);
/* Hand over finished episodes: episode e = (ep_game[e], ep_bank[e]) (dev int32) with T_e moves is copied to
 * rows [step_off[e], step_off[e] + T_e) of out_action/out_reward/out_root/out_visits, to rows
 * [step_off[e] + e*stack, +stack + T_e) of out_obs and [step_off[e] + e, +T_e + 1) of out_legal (dev
 * int64 step_off = exclusive prefix sum of the T_e); the bank is freed. */
int hz_traj_pack(void* stream, const hz_traj_view* v, int num_episodes, const int32_t* ep_game, const int32_t* ep_bank,
                 const int64_t* step_off, uint8_t* out_obs, uint8_t* out_legal, int32_t* out_action,
                 int32_t* out_reward, int32_t* out_visits, float* out_root);
/* Policy targets from visit counts (store_search_stats, game.py:194-197; the reanalyze caller,
 * /root/reference/core/reanalyze_worker.py:352-367, SURVEY.md §8f N4): out[i][a] = visits[i][a] / sum_a visits[i]
 * as a correctly rounded double quotient (Python's int / int, the sum taken in 64 bits), rows with mask[i] == 0
 * (dev uint8[N], NULL = keep all) all zero.  A kept row whose counts sum to 0 is all NaN (0 / 0: Python raises
 * ZeroDivisionError there); SearchConfig rejects num_simulations < 2, so no search leaves such a root.
 * out64 double[N][A] and/or out32 float[N][A] (dev). */
int hz_visit_policy(void* stream, const int32_t* visits, const uint8_t* mask, int num, int num_actions, double* out64,
                    float* out32);

/* A fixed chain of nn.Linear-shaped GEMMs executed with cuBLASLt, one launch each:
 *   D[m][n] = act( A[m][k] . W[n][k]^T + bias[n] + C[m][n] ),  all row-major, strided batches allowed.
 * Pointers are captured at creation (static buffers: the chain is CUDA-graph friendly); hz_gemm_plan_set_operand
 * re-points single operands. */
typedef struct hz_gemm_step {
  const void* a;    int64_t lda; int64_t stride_a;     /* activations */
  const void* w;    int64_t ldw; int64_t stride_w;     /* weights in nn.Linear layout [n][k] */
  const void* bias; int64_t stride_bias;               /* [n] or NULL */
  const void* c;    int64_t ldc; int64_t stride_c;     /* residual or NULL */
  void* d;          int64_t ldd; int64_t stride_d;     /* output */
  int32_t m, n, k, batch, relu;
} hz_gemm_step;
typedef struct hz_gemm_plan hz_gemm_plan;
int hz_gemm_plan_create(hz_gemm_plan** out, int device, int elem_bytes, const hz_gemm_step* steps, int n_steps); /* sync */
int hz_gemm_plan_destroy(hz_gemm_plan* p);                                                                     /* sync */
int hz_gemm_plan_steps(const hz_gemm_plan* p);
/* Re-point one operand of one step (which: 0 = A, 1 = C, 2 = D) at another buffer of the same shape and leading
 * dimension, 256-byte aligned.  Takes effect for the following hz_gemm_plan_run calls (and is what a CUDA graph
 * captures): the search loop makes the dynamics network write each new hidden state straight into pool[x]. */
int hz_gemm_plan_set_operand(hz_gemm_plan* p, int step, int which, void* ptr);
/* Size every step's library kernel for `sm_count` SMs instead of the whole device (CUBLASLT_MATMUL_DESC_SM_COUNT_TARGET;
 * 0 = whole device, the default): the heuristic picks fewer, fatter CTAs, so the GEMMs of several plans running on
 * different streams — independent searches in flight — share the GPU instead of queueing behind one another's
 * grid-filling launches.  Re-selects the kernels at once; call before capturing the plan in a CUDA graph. */
int hz_gemm_plan_set_sm_target(hz_gemm_plan* p, int sm_count);
/* cuBLASLt launches issued through hz_gemm_plan_run in this process (library GEMMs, counted apart from
 * hz_launch_count, which counts this library's own kernels) */
int64_t hz_gemm_launch_count(void);
int hz_gemm_plan_run(hz_gemm_plan* p, void* stream, int first, int count);

/* Row-block resident executor of the recurrent_inference chain (fp16): the same function as the hz_gemm_plan that
 * hanabizero_b200/plan.py builds (seven steps for MuZeroNetFull, five for MuZeroNet / Hanabi-Small;
 * /root/reference/core/model.py:74-84, config/hanabi_control/model.py:199-216,301-318, eval mode, BatchNorm folded),
 * as ONE launch in which each CTA keeps 128 rows of the batch in shared memory / TMEM through all layers and only the
 * weights stream in (TMA + tcgen05, hanabizero_b200/csrc/hz_rowchain.cu).  A 4096-row batch occupies 32 SMs, which is
 * what several searches in flight want.  hz_rowchain_create builds the Hanabi-Full chain, hz_rowchain_create_small the
 * Hanabi-Small one; every other hz_rowchain_* call serves both.  All pointers dev, fp16, 16-byte aligned, captured at
 * creation. */
typedef struct hz_rowchain_weights {
  const void* w1;  int64_t ld_w1;     /* [512][ld_w1]: fc1 (+bn1) over [state | one-hot action] */
  const void* w1a_t;                  /* [onehot_cols][512]: the action columns of w1, transposed */
  const void* b1;
  const void* w2;  const void* b2;    /* [512][512] */
  const void* w3;  const void* b3;    /* [512][512]; the residual is the input state */
  const void* wh1; const void* bh1;   /* [768][512]: first layers of policy | value | reward heads */
  const void* wb2; const void* bb2;   /* [3][256][256]: second layers, same order */
  const void* wa2; const void* ba2;   /* [256][256]: policy residual block, second layer */
  const void* wb3; const void* bb3;   /* [3][logit_cols][256]: output layers value | reward | policy */
  int32_t state_cols, head_cols, onehot_cols, logit_cols;   /* 512, 256, 32, <= 256 (multiple of 16) */
} hz_rowchain_weights;   /* shapes as hz_rowchain_create takes them; hz_rowchain_create_small states its own */
typedef struct hz_rowchain hz_rowchain;
/* x0 [rows][ld_x0] = state | one-hot(action) (what hz_trees_search_step hands over), state [rows][512] receives the
 * next hidden state, out_logits [3][rows][logit_cols] = value | reward | policy logits. */
int hz_rowchain_create(hz_rowchain** out, int device, const hz_rowchain_weights* w, int rows, const void* x0,
                       int64_t ld_x0, void* state, void* out_logits);                                   /* sync */
/* Hanabi-Small (MuZeroNet): fc1's skip s joins after bn1, no residual after fc3, one layer per head.  Same struct:
 * state_cols 512, head_cols 128, onehot_cols 16, logit_cols 64; w1 [512][ld_w1 >= 528], w1a_t [16][512],
 * wh1 [384][512] = first layers of value | reward | policy heads, wb3 [3][64][128] = their output layers (same order);
 * wb2 / bb2 / wa2 / ba2 must be NULL.  x0 [rows][ld_x0 >= 528], out_logits [3][rows][64]. */
int hz_rowchain_create_small(hz_rowchain** out, int device, const hz_rowchain_weights* w, int rows, const void* x0,
                             int64_t ld_x0, void* state, void* out_logits);                             /* sync */
int hz_rowchain_destroy(hz_rowchain* e);
/* Re-point the next-state output (the search loop passes pool[x]); takes effect for the following runs. */
int hz_rowchain_set_state(hz_rowchain* e, void* state);
int hz_rowchain_run(hz_rowchain* e, void* stream);
int hz_rowchain_grid(const hz_rowchain* e);                     /* CTAs per launch */
/* Debug: per-CTA globaltimer stamps of the first row block, uint64[grid][10 phase slots][4] (Hanabi-Full runs 10
 * phases, Hanabi-Small 6) =
 * {MMA may start, MMAs issued, accumulators complete, tile written back}. */
int hz_rowchain_set_trace(hz_rowchain* e, int enable);
int hz_rowchain_read_trace(hz_rowchain* e, uint64_t* host_out, int64_t count);                          /* sync */

/* ------------------------------------------------------------------------------------------
 * Search waves: `count` independent root batches ("tickets") of n roots each searched as ONE batch of slots * n trees
 * (hanabizero_b200/mcts.py SearchPipeline(wave=slots); the reference's actors each submit their own p_mcts_num roots,
 * core/selfplay_worker.py:93-102).  Ticket k owns rows [k*n, (k+1)*n) of the wave.  Every pointer of the table and
 * every buffer is device memory of `device` or page-locked host memory (read and written by the kernel itself under
 * unified addressing, as hz_envs_host_step does); anything else (pageable host memory, another device's memory), a
 * misaligned pointer (16 bytes for hidden, 4 for the rest), count outside 1..slots, slots outside 1..64, num_actions
 * outside 1..32, n < 1, slots * n > 2^24 or hidden_row_bytes not a multiple of 16 in 16..65536 is HZ_ERR_ARG, checked
 * before anything is launched.  The table is passed to the kernel by value: it may be reused as soon as the call
 * returns.  Both calls are one launch and asynchronous; the ticket buffers must stay valid until the stream gets there.
 * ------------------------------------------------------------------------------------------ */
typedef struct hz_wave_ticket {
  const float* noise;      /* [n][A] or NULL (= zeros) */
  const float* reward;     /* [n] */
  const float* logits;     /* [n][A] */
  const int32_t* legal;    /* [n][A] */
  const void* hidden;      /* [n][hidden_row_bytes] */
  int32_t* out_visits;     /* [n][A] or NULL (hz_wave_unpack only) */
  float* out_values;       /* [n] or NULL (hz_wave_unpack only) */
} hz_wave_ticket;
/* Fills the wave's staging buffers (slots * n rows, the inputs of hz_trees_prepare and of the search's hidden-state
 * pool): ticket k's rows go to rows [k*n, (k+1)*n); the rows of slots count..slots-1 become padding roots with zero
 * noise, reward, logits and hidden state and an all-zero legal mask (a root without children), so a partial wave runs
 * the full-size search unchanged.  noise == NULL (a wave prepared without noise) leaves the noise rows unwritten. */
int hz_wave_pack(void* stream, int device, const hz_wave_ticket* tickets, int count, int slots, int n, int num_actions,
                 int hidden_row_bytes, float* noise, float* reward, float* logits, int32_t* legal, void* hidden);
/* Scatters the wave's root statistics, laid out as hz_trees_root_stats writes them into one int32 buffer
 * stats = [slots*n*A visit counts | slots*n value bit patterns], to every ticket's out_visits / out_values (NULL = not
 * wanted).  `slots` is the wave's size, which places the value block. */
int hz_wave_unpack(void* stream, int device, const hz_wave_ticket* tickets, int count, int slots, int n,
                   int num_actions, const int32_t* stats);
/* Policy targets straight from a wave's statistics (the reanalyze caller, SearchPipeline.submit_observations with
 * out_policy): for ticket k, out[i][a] = visits[k*n + i][a] / sum_a visits[k*n + i] as hz_visit_policy computes it
 * (correctly rounded double quotient; all zero where mask[i] == 0, mask == NULL keeps every row), visits being the first
 * slots*n*A words of `stats` (laid out as for hz_wave_unpack).  mask uint8 [n] and out double [n][A] (8-byte aligned,
 * never NULL) are device memory of `device` or page-locked host memory, read and written by the kernel itself.  Sizes
 * and pointers are checked before the launch as in hz_wave_unpack; one launch, the table travels by value. */
typedef struct hz_policy_ticket {
  const uint8_t* mask;     /* [n] or NULL */
  double* out;             /* [n][A] */
} hz_policy_ticket;
int hz_wave_policy(void* stream, int device, const hz_policy_ticket* tickets, int count, int slots, int n,
                   int num_actions, const int32_t* stats);

/* Observation tickets (SearchPipeline.submit_observations): a wave whose tickets hand in stacked observations instead
 * of the representation network's outputs.  hz_obs_pack fills, for ticket k, rows [k*n, (k+1)*n) of
 *   x      [slots*n][stack * frame_stride] half (elem_bytes 2) or float (4), 16-byte aligned: the root inference's input
 *          as hz_ring_gather writes it — frame j (oldest first) at column j * frame_stride, padding columns 0;
 *   legal  int32 [slots*n][A], the mask hz_trees_prepare takes (int32 masks as given, the others as 0 / 1);
 *   noise  float [slots*n][A], or NULL for a wave prepared without noise (a ticket's NULL noise gives zeros).
 * The rows of slots count..slots-1 are padding roots: zero input and an all-zero legal mask, as in hz_wave_pack.
 * Frame formats of a ticket's obs, row i at obs + i * ld_obs elements, frame j of the row at j * D (j * W for bits):
 *   HZ_OBS_F32   float   [n][stack][D] values, converted to x's type
 *   HZ_OBS_U8    uint8   [n][stack][D] values (0/1 bytes: HanabiVecEnv(obs_dtype=torch.uint8), the recorder's rows)
 *   HZ_OBS_BITS  uint32  [n][stack][W] packed strings: the frame is bits [bit_offset, bit_offset + D), bit b in word
 *                b / 32 at position b % 32 (hz_envs_step_observe_bits' order; bit_offset 0 = the global observation,
 *                own_len = its local suffix)
 * Legal formats, row i at legal + i * ld_legal elements: HZ_LEGAL_I32 int32 [n][A] and HZ_LEGAL_F32 float [n][A]
 * (non-zero = legal), HZ_LEGAL_MASK one uint32 per root, bit a = action a legal (word 0 of the meta rows
 * hz_envs_step_observe_bits / hz_envs_host_step write: ld_legal 4).  Pointers: device memory of `device` or
 * page-locked host memory, which the kernel reads itself; 4-byte aligned except uint8 frames.  Sizes as hz_wave_pack,
 * plus: stack 1..64, 1 <= D <= frame_stride, frame_stride a multiple of 16, stack * frame_stride <= 65536, and for bit
 * frames W >= 1 with bit_offset + D <= 32 W.  Everything is checked before the launch (HZ_ERR_ARG).  One launch,
 * asynchronous; the table and layout may be reused when the call returns, the sources must stay valid until the stream
 * gets there.  Results go back through hz_wave_unpack with only out_visits / out_values set. */
enum { HZ_OBS_F32 = 0, HZ_OBS_U8 = 1, HZ_OBS_BITS = 2 };
enum { HZ_LEGAL_I32 = 0, HZ_LEGAL_F32 = 1, HZ_LEGAL_MASK = 2 };
typedef struct hz_obs_ticket {
  const void* obs;         /* frames, `obs_format` */
  int64_t ld_obs;          /* row stride in elements of the format (floats, bytes, words) */
  const void* legal;       /* legal moves, `legal_format` */
  int64_t ld_legal;        /* row stride in elements (int32 / float / mask words) */
  const float* noise;      /* [n][A] contiguous, or NULL (= zeros) */
  int32_t obs_format;      /* HZ_OBS_* */
  int32_t legal_format;    /* HZ_LEGAL_* */
} hz_obs_ticket;
typedef struct hz_obs_layout {
  int32_t stack;           /* frames per root */
  int32_t frame_dim;       /* D: values per frame */
  int32_t frame_stride;    /* columns per frame in x */
  int32_t elem_bytes;      /* x: 2 = half, 4 = float */
  int32_t frame_words;     /* W: words per packed frame (HZ_OBS_BITS) */
  int32_t bit_offset;      /* first bit of the frame in its packed string (HZ_OBS_BITS) */
} hz_obs_layout;
int hz_obs_pack(void* stream, int device, const hz_obs_ticket* tickets, int count, int slots, int n, int num_actions,
                const hz_obs_layout* layout, void* x, int32_t* legal, float* noise);
/* hz_obs_pack over frame WINDOWS (the reanalyze batch: consecutive positions of one trajectory share frames): row i of
 * a ticket's obs holds stack + positions - 1 consecutive frames in any of the three formats (ld_obs = the window row
 * stride, at least the window's elements), and root r = i * positions + p takes window frames p .. p + stack - 1,
 * oldest first, landing in x exactly where hz_obs_pack puts root r of the expanded stacks.  Legal rows and noise stay
 * per root (n rows).  positions is 1..n and divides n.  Everything else as hz_obs_pack, checked before the launch. */
int hz_obs_pack_windows(void* stream, int device, const hz_obs_ticket* tickets, int count, int slots, int n,
                        int num_actions, const hz_obs_layout* layout, int positions, void* x, int32_t* legal,
                        float* noise);
/* hz_obs_pack_windows with the windows read from an episode store (hanabizero_b200/trajectory.py EpisodeStore): byte
 * frame rows of D = frame_dim values in `frames` (row stride ld_frames bytes) and legal rows of num_actions 0/1 bytes in
 * `legal`, as hz_traj_pack writes them.  Sample i of a ticket (roots i * positions .. i * positions + positions - 1) is
 * four int32 in samples[i]: {first frame row of its window, last frame row of its episode, legal row of its first
 * position, number of positions with targets c (0..positions)}.  Root r = i * positions + p takes frame rows
 * min(first + p + j, last) for j = 0..stack-1, legal row first_legal + p and its noise where p < c (noise entries whose
 * legal byte is 0 become 0), an all-zero legal row and noise where p >= c, and mask[r] = p < c — the mask that
 * hz_wave_policy takes for the ticket's targets.  frames, legal, samples (16-byte aligned), noise and mask: device
 * memory of `device` or page-locked host memory, read and written by the kernel itself; only mask may not be NULL among
 * the outputs, noise may (zeros).  The rows the samples name are not checked: they must lie in the arenas.  Everything
 * else as hz_obs_pack_windows, checked before the launch; one launch, the table (48 bytes a ticket) travels by value. */
typedef struct hz_obs_episode_ticket {
  const uint8_t* frames;   /* frame arena */
  int64_t ld_frames;       /* bytes per frame row (>= frame_dim) */
  const uint8_t* legal;    /* legal arena [rows][num_actions] */
  const int32_t* samples;  /* [n / positions][4] */
  const float* noise;      /* [n][A] contiguous, or NULL (= zeros) */
  uint8_t* mask;           /* [n] out */
} hz_obs_episode_ticket;
int hz_obs_pack_episodes(void* stream, int device, const hz_obs_episode_ticket* tickets, int count, int slots, int n,
                         int num_actions, const hz_obs_layout* layout, int positions, void* x, int32_t* legal,
                         float* noise);

#ifdef __cplusplus
}
#endif
#endif /* HZB200_H */
