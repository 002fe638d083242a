// Batched Hanabi environment for sm_100a: one warp per game.
//
// Replaces, for the two presets the reference uses (rl_env.py:110-131, both 2-player, 5 ranks),
// the C++ Hanabi Learning Environment behind libpyhanabi.so as sequenced by HanabiEnv.reset/step:
//   rules     hanabi_state.cc:104-275 (ApplyMove, legality, fireworks, tokens, AdvanceToNextPlayer)
//   hands     hanabi_hand.cc:80-126   (AddCard, RemoveFromHand, RevealColor/RevealRank knowledge)
//   deals     hanabi_state.cc:277-325 + hanabi_game.cc:106-112: std::discrete_distribution over
//             count/deck_size with the game's std::mt19937 (libstdc++ algorithm restated in fp64)
//   observer  hanabi_observation.cc:52-96, encoder canonical_encoders.cc:66-486
//   glue      rl_env.py:254-263,426-442 (global = own hand ‖ encoding ‖ turn; local; legal mask;
//             reward = score delta; done)
//
// HBM layout: state [N][128] bytes (one 128-byte line per game, loaded as one word per lane into
// shared memory), mt [N][624] uint32 + mti [N] (the game-owned Mersenne Twister, persists across
// resets).  Observations are written lane-strided (coalesced) as float 0/1.  Scalar game logic is
// executed by lane 0 on the shared-memory copy; the deal distribution (<= 25 outcomes), the
// twister refill, legality and the 785/660-wide encodings are lane-parallel.
#include "hz_common.cuh"

namespace hz {

#ifdef HZ_TRACE
// debug build only: per-game cycle stamps of the env kernel's phases (scripts/exp_env_trace.py)
__device__ long long* g_env_trace = nullptr;
#define HZ_ESTAMP(k) do { if (g_env_trace && lane == 0) g_env_trace[(size_t)gi * 16 + (k)] = clock64(); } while (0)
#define HZ_DSTAMP(k) do { if (g_env_trace && lane == 0) { const long long _c = clock64(); g_env_trace[(size_t)dgi * 16 + 10 + (k)] += _c - dt0; dt0 = _c; } } while (0)
#else
#define HZ_ESTAMP(k) do { } while (0)
#define HZ_DSTAMP(k) do { } while (0)
#endif

constexpr int kEnvWarps = 4;
constexpr int kStateBytes = 128;
constexpr int P = 2;  // both reference presets are 2-player

// byte offsets inside the 128-byte game state
enum : int {
  O_CUR = 0, O_NEXT = 1, O_INFO = 2, O_LIFE = 3, O_DECK = 4, O_TURNS = 5,
  O_LMVALID = 6, O_LMTYPE = 7, O_LMPLAYER = 8, O_LMIDX = 9, O_LMTGT = 10, O_LMCOLOR = 11,
  O_LMRANK = 12, O_LMCARD = 13, O_LMFLAGS = 14, O_LMREVEAL = 15,
  O_FW = 16,       // [5]
  O_HLEN = 21,     // [2]
  O_DECKCNT = 24,  // [25]
  O_DISC = 49,     // [25]
  O_HAND = 74,     // [2][5][5] = {card, colour mask, rank mask, hinted colour, hinted rank}
};
enum : int { MV_PLAY = 1, MV_DISCARD = 2, MV_REVEAL_COLOR = 3, MV_REVEAL_RANK = 4 };  // hanabi_move.h:33
constexpr uint8_t kNone = 0xff;

struct Rules {
  int C, R, H, max_info, max_life, A, enc_len, own_len, deck_max;
};

__device__ __forceinline__ int hand_off(int p, int k) { return O_HAND + (p * 5 + k) * 5; }
__device__ __forceinline__ int instances(int rank, int R) { return rank == 0 ? 3 : (rank == R - 1 ? 1 : 2); }

// ---- std::mt19937 (game-owned; hanabi_game.h:114) -------------------------------------------------
__device__ __forceinline__ void mt_refill(uint32_t* mt, int lane) {
  // in-place block update, 32 elements per pass: every element k needs old mt[k], old mt[k+1]
  // (new mt[0] for k = 623) and mt[k+397 mod 624], which is old for k < 227 and was rewritten at
  // least 7 passes earlier otherwise.  Reads of a pass complete before its writes.
  for (int base = 0; base < 624; base += HZ_WARP) {
    const int k = base + lane;
    uint32_t v = 0;
    if (k < 624) {
      const uint32_t a = mt[k], b = mt[k == 623 ? 0 : k + 1], c = mt[k < 227 ? k + 397 : k - 227];
      const uint32_t y = (a & 0x80000000u) | (b & 0x7fffffffu);
      v = c ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
    __syncwarp();
    if (k < 624) mt[k] = v;
    __syncwarp();
  }
}

// The next 32 raw state words are fetched once per kernel (one coalesced load, lane i holds
// mt[start + i]); draws inside that window come from a shuffle instead of a dependent global load.
struct MtWindow {
  uint32_t word;   // this lane's prefetched state word
  int start;       // index of lane 0's word; < 0 once a refill invalidated the window
};

__device__ __forceinline__ MtWindow mt_prefetch(const uint32_t* mt, int mti, int lane) {
  MtWindow w;
  w.start = mti;
  w.word = (mti + lane < 624) ? mt[mti + lane] : 0u;
  return w;
}

__device__ __forceinline__ uint32_t mt_draw(uint32_t* mt, int& mti, MtWindow& win, int lane) {
  if (mti >= 624) {
    mt_refill(mt, lane);
    mti = 0;
    win.start = -1;
  }
  uint32_t z;
  const int off = mti - win.start;
  if (win.start >= 0 && off >= 0 && off < HZ_WARP) {   // warp-uniform
    z = __shfl_sync(HZ_FULL, win.word, off);
  } else {
    z = mt[mti];
  }
  ++mti;
  z ^= (z >> 11);
  z ^= (z << 7) & 0x9d2c5680u;
  z ^= (z << 15) & 0xefc60000u;
  z ^= (z >> 18);
  return z;
}

__device__ __forceinline__ int player_to_deal(const uint8_t* st, int H) {  // hanabi_state.cc:157-164
  if (st[O_HLEN] < H) return 0;
  if (st[O_HLEN + 1] < H) return 1;
  return -1;
}

__device__ __forceinline__ void advance(uint8_t* st, int H) {  // hanabi_state.cc:104-111
  if (st[O_DECK] > 0 && player_to_deal(st, H) >= 0) {
    st[O_CUR] = kNone;
  } else {
    st[O_CUR] = st[O_NEXT];
    st[O_NEXT] = (uint8_t)((st[O_CUR] + 1) % P);
  }
}

// ApplyRandomChance (hanabi_state.cc:282-286): ChanceOutcomes (313-325) -> PickRandomChance
// (hanabi_game.cc:106-112, libstdc++ discrete_distribution + generate_canonical<double,53>) ->
// ApplyMove(kDeal) (221-243).  Warp-cooperative; all lanes must call.  scratch: 64 doubles of shared
// memory per warp.  The two ordered fp64 sums (std::accumulate, std::partial_sum) are evaluated in
// libstdc++'s order over ALL NT card types instead of the compacted outcome list: a type the deck no
// longer holds contributes +0.0, and adding +0.0 to a non-negative double is exact, so the bits are
// the same — but the trip counts are compile-time constants, the loops unroll, the operand loads
// leave the add chain, and there is no divergence.  (A finished game re-deals ten cards inside the
// launch: these chains are the tail of the kernel.)
template <int NT>
__device__ __forceinline__ void deal_random(uint8_t* st, const Rules& g, uint32_t* mt, int& mti, MtWindow& win,
                                            double* scratch, int lane, int dgi = 0) {
#ifdef HZ_TRACE
  long long dt0 = clock64();
  if (g_env_trace && lane == 0) g_env_trace[(size_t)dgi * 16 + 9] += 16;
#endif
  const int cnt = lane < NT ? st[O_DECKCNT + lane] : 0;
  const bool have = cnt > 0;
  const unsigned mask = __ballot_sync(HZ_FULL, have);
  const int m = __popc(mask);
  int pick = __ffs(mask) - 1;  // single outcome: _M_prob.size() < 2 -> index 0, no draw consumed
  if (m >= 2) {
    double* w = scratch;        // [32] ChanceOutcomeProb per card type (0.0 where the deck holds none)
    double* qn = scratch + 32;  // [32] normalised
    const double wv = have ? __ddiv_rn((double)cnt, (double)st[O_DECK]) : 0.0;
    w[lane] = wv;
    __syncwarp();
    HZ_DSTAMP(0);
    double sum = 0.0;  // std::accumulate ascending
#pragma unroll
    for (int i = 0; i < NT; ++i) sum = __dadd_rn(sum, w[i]);
    HZ_DSTAMP(1);
    qn[lane] = have ? __ddiv_rn(wv, sum) : 0.0;  // __normalize
    __syncwarp();
    HZ_DSTAMP(2);
    double acc = 0.0;  // std::partial_sum ascending, this lane's prefix
#pragma unroll
    for (int i = 0; i < NT; ++i) acc = __dadd_rn(acc, i <= lane ? qn[i] : 0.0);
    // lanes without an outcome never match; _M_cp.back() = 1.0
    HZ_DSTAMP(3);
    const double cp = !have ? 2.0 : (lane == 31 - __clz(mask) ? 1.0 : acc);
    const uint32_t u0 = mt_draw(mt, mti, win, lane);
    const uint32_t u1 = mt_draw(mt, mti, win, lane);
    double p = __dadd_rn((double)u0, __dmul_rn((double)u1, 4294967296.0));
    p = __dmul_rn(p, 5.421010862427522170037264004349708557128906250e-20);  // / 2^64 (exact)
    if (p >= 1.0) p = 0x1.fffffffffffffp-1;                                // nextafter(1, 0)
    const unsigned ge = __ballot_sync(HZ_FULL, have && cp >= p);           // std::lower_bound
    pick = __ffs(ge) - 1;
    __syncwarp();
    HZ_DSTAMP(4);
  }
  if (lane == 0) {
    const int to = player_to_deal(st, g.H);
    const int k = st[O_HLEN + to]++;
    const int o = hand_off(to, k);
    st[o] = (uint8_t)pick;
    st[o + 1] = (uint8_t)((1 << g.C) - 1);
    st[o + 2] = (uint8_t)((1 << g.R) - 1);
    st[o + 3] = kNone;
    st[o + 4] = kNone;
    st[O_DECKCNT + pick]--;
    st[O_DECK]--;
    advance(st, g.H);
  }
  __syncwarp();
  HZ_DSTAMP(5);
}

// LegalMoves (hanabi_state.cc:288-304, MoveIsLegal 166-219) for all move uids at once, as a bit mask (warp-uniform):
// lanes first agree on which colours / ranks the partner's hand holds, then each lane tests its own move id.
// No terminal check, like the reference (the mask is non-zero at terminal states).  cur < 0 (chance node): no move.
__device__ __forceinline__ unsigned legal_mask(const uint8_t* st, const Rules& g, int lane) {
  const int cur = (int8_t)st[O_CUR];
  if (cur < 0) return 0u;
  const int H = g.H, C = g.C, R = g.R;
  const int other = (cur + 1) % P, n_me = st[O_HLEN + cur], n_ot = st[O_HLEN + other];
  const int card = lane < n_ot ? st[hand_off(other, lane)] : -1;
  const unsigned cmask = __reduce_or_sync(HZ_FULL, card >= 0 ? 1u << (card / R) : 0u);
  const unsigned rmask = __reduce_or_sync(HZ_FULL, card >= 0 ? 1u << (card % R) : 0u);
  bool ok = false;
  if (lane < g.A) {
    if (lane < H) ok = st[O_INFO] < g.max_info && lane < n_me;                       // discard
    else if (lane < 2 * H) ok = lane - H < n_me;                                     // play
    else if (lane < 2 * H + C) ok = st[O_INFO] > 0 && ((cmask >> (lane - 2 * H)) & 1u);       // reveal colour
    else ok = st[O_INFO] > 0 && ((rmask >> (lane - 2 * H - C)) & 1u);                         // reveal rank
  }
  return __ballot_sync(HZ_FULL, ok);
}

// HanabiState::ApplyMove for a player move (hanabi_state.cc:221-275), warp-cooperative (all lanes call): the hand
// shift of RemoveFromHand (hanabi_hand.cc:87-94) moves one byte per lane, RevealColor / RevealRank
// (hanabi_hand.cc:96-126) update one card per lane, lane 0 keeps the scalar book-keeping.
__device__ __forceinline__ void apply_move(uint8_t* st, const Rules& g, int uid, int lane) {
  const int H = g.H, R = g.R, me = (int8_t)st[O_CUR];
  const int t = (me + 1) % P;
  // ---- read phase: everything any lane needs, before anyone writes
  const int deck = st[O_DECK], info = st[O_INFO];
  const bool is_discard = uid < H, is_play = !is_discard && uid < 2 * H;
  const int k = is_discard ? uid : uid - H;                       // hand slot of a discard / play
  const int n_me = st[O_HLEN + me], n_t = st[O_HLEN + t];
  const int c = (is_discard || is_play) ? st[hand_off(me, k)] : 0;
  // RemoveFromHand: byte j of the mover's hand takes the byte one card further once j is at or past slot k
  const int hb = O_HAND + me * 5 * 5;
  uint8_t moved = 0;
  const bool shift = (is_discard || is_play) && lane < 25 && lane >= 5 * k && lane + 5 < 5 * n_me;
  if (shift) moved = st[hb + lane + 5];
  // Reveal*: lane = card slot of the target hand
  const bool is_color = !is_discard && !is_play && uid < 2 * H + g.C;
  const int hint = is_color ? uid - 2 * H : uid - 2 * H - g.C;
  bool match = false;
  int ko = 0;
  uint8_t know_mask = 0;
  if (!is_discard && !is_play && lane < n_t) {
    ko = hand_off(t, lane);
    const int card = st[ko];
    match = (is_color ? card / R : card % R) == hint;
    know_mask = st[ko + (is_color ? 1 : 2)];
  }
  const unsigned reveal = __ballot_sync(HZ_FULL, match);
  const int fw = is_play ? st[O_FW + c / R] : 0;
  __syncwarp();
  // ---- write phase
  if (shift) st[hb + lane] = moved;
  if (!is_discard && !is_play && lane < n_t) {
    if (match) {
      st[ko + (is_color ? 3 : 4)] = (uint8_t)hint;
      st[ko + (is_color ? 1 : 2)] = (uint8_t)(1 << hint);
    } else {
      st[ko + (is_color ? 1 : 2)] = know_mask & (uint8_t)~(1 << hint);
    }
  }
  if (lane == 0) {
    if (deck == 0) st[O_TURNS]--;
    st[O_LMVALID] = 1;
    st[O_LMPLAYER] = (uint8_t)me;
    st[O_LMIDX] = kNone; st[O_LMTGT] = kNone; st[O_LMCOLOR] = kNone; st[O_LMRANK] = kNone;
    st[O_LMCARD] = kNone; st[O_LMREVEAL] = 0;
    uint8_t flags = 0;
    if (is_discard) {
      st[O_LMTYPE] = MV_DISCARD;
      st[O_LMIDX] = (uint8_t)k;
      if (info < g.max_info) { st[O_INFO] = (uint8_t)(info + 1); flags |= 2; }
      st[O_LMCARD] = (uint8_t)c;
      st[O_DISC + c]++;
      st[O_HLEN + me] = (uint8_t)(n_me - 1);
    } else if (is_play) {
      st[O_LMTYPE] = MV_PLAY;
      st[O_LMIDX] = (uint8_t)k;
      st[O_LMCARD] = (uint8_t)c;
      const int col = c / R, rk = c % R;
      if (rk == fw) {  // AddToFireworks hanabi_state.cc:132-144
        st[O_FW + col] = (uint8_t)(fw + 1);
        flags |= 1;
        if (fw + 1 == R && info < g.max_info) { st[O_INFO] = (uint8_t)(info + 1); flags |= 2; }
      } else {
        st[O_LIFE]--;
        st[O_DISC + c]++;
      }
      st[O_HLEN + me] = (uint8_t)(n_me - 1);
    } else {
      st[O_LMTGT] = 1;
      st[O_INFO] = (uint8_t)(info - 1);
      st[O_LMTYPE] = is_color ? MV_REVEAL_COLOR : MV_REVEAL_RANK;
      st[is_color ? O_LMCOLOR : O_LMRANK] = (uint8_t)hint;
      st[O_LMREVEAL] = (uint8_t)reveal;
    }
    st[O_LMFLAGS] = flags;
  }
  __syncwarp();
  if (lane == 0) advance(st, H);
}

__device__ __forceinline__ int score_of(const uint8_t* st, int C) {  // hanabi_state.cc:359-364
  if (st[O_LIFE] == 0) return 0;
  int s = 0;
  for (int c = 0; c < C; ++c) s += st[O_FW + c];
  return s;
}

__device__ __forceinline__ bool is_terminal(const uint8_t* st, const Rules& g) {  // hanabi_state.cc:366-377
  return st[O_LIFE] < 1 || score_of(st, g.C) >= g.C * g.R || (int8_t)st[O_TURNS] <= 0;
}

// HanabiState ctor (hanabi_state.cc:90-102) + HanabiDeck (53-64); lanes cooperate
__device__ __forceinline__ void new_state(uint8_t* st, const Rules& g, int lane) {
  for (int i = lane; i < kStateBytes; i += HZ_WARP) st[i] = 0;
  __syncwarp();
  if (lane < g.C * g.R) st[O_DECKCNT + lane] = (uint8_t)instances(lane % g.R, g.R);
  if (lane == 0) {
    st[O_CUR] = kNone;
    st[O_NEXT] = 0;  // GetSampledStartPlayer with random_start_player = false
    st[O_INFO] = (uint8_t)g.max_info;
    st[O_LIFE] = (uint8_t)g.max_life;
    st[O_DECK] = (uint8_t)g.deck_max;
    st[O_TURNS] = P;
  }
  __syncwarp();
}

// ---- observation as a bit string ---------------------------------------------------------------
// The global observation (rl_env.py:262,433) = EncodeOwnHand (canonical_encoders.cc:465-486) ‖
// CanonicalObservationEncoder::Encode (441-463: hands 66-109, board 127-171, discards 192-215, last
// action 240-342, card knowledge 370-423) ‖ turn one-hot (rl_env.py:256-257).  It is assembled as
// ~44 bit-field segments OR-ed into shared-memory words (one or two segments per lane), then expanded
// to float 0/1 with coalesced stores; the local observation is its suffix.
__device__ __forceinline__ void or_bits(uint32_t* w, int bit, uint32_t v) {
  if (v == 0u) return;
  const int i = bit >> 5, sh = bit & 31;
  atomicOr(&w[i], v << sh);
  if (sh != 0 && (v >> (32 - sh)) != 0u) atomicOr(&w[i + 1], v >> (32 - sh));
}
__device__ __forceinline__ uint32_t ones(int n) { return n >= 32 ? 0xffffffffu : ((1u << n) - 1u); }

template <int C, int R, int H, int MI, int ML>
struct ObsLayout {
  static constexpr int BPC = C * R, OWN = H * BPC;
  static constexpr int PER_COLOR = 3 + 2 * (R - 2) + 1, DECK_MAX = PER_COLOR * C;
  static constexpr int HANDS = (P - 1) * H * BPC, DW = DECK_MAX - P * H;
  static constexpr int LAST_A = P + 4 + P + C + R + H + H, LAST = LAST_A + BPC + 2, PER_CARD = BPC + C + R;
  static constexpr int o_hands = OWN, o_miss = o_hands + HANDS, o_deck = o_miss + P, o_fw = o_deck + DW;
  static constexpr int o_info = o_fw + BPC, o_life = o_info + MI, o_disc = o_life + ML, o_last = o_disc + DECK_MAX;
  static constexpr int o_know = o_last + LAST, o_turn = o_know + P * H * PER_CARD, GLOBAL = o_turn + P;
  static constexpr int ENC = GLOBAL - OWN - P, WORDS = (GLOBAL + 31) / 32 + 1;
  static_assert(DW <= 64 && LAST_A <= 32 && BPC + 2 <= 32 && PER_COLOR <= 32, "segment wider than a word");
  static_assert(2 * H + P * H + C + 1 <= 32, "one lane per segment");
};

// Every lane prepares at most two (bit offset, value) fields from the game state — the part that differs from lane to
// lane is plain byte loads and ALU work — and the shared-memory atomics that OR the fields into the bit string are
// issued afterwards by uniform code, all lanes at once (a per-lane switch around the atomics serialises their ~60-cycle
// round trips branch after branch):
//   lanes [0, 2H)         one hand card each (own hand, then the partner's)  + one board field each:
//                         fireworks, "hand is short" bits, deck (two words), information / life tokens, turn
//   lanes [2H, 2H + P*H)  card knowledge of one (player, slot): plausible-card grid + hinted colour / rank
//   next C lanes          discards of one colour
//   one more lane         the last move (two fields)
template <int C, int R, int H, int MI, int ML>
__device__ __forceinline__ void obs_build(const uint8_t* st, int cur, uint32_t* w, int lane) {
  using L = ObsLayout<C, R, H, MI, ML>;
  static_assert(2 * H >= 7 || H == 2, "board fields ride on the hand lanes");
  const int other = (cur + 1) % P;
  int bit0 = 0, bit1 = 0;
  uint32_t v0 = 0, v1 = 0;
  if (lane < 2 * H) {
    // hands (canonical_encoders.cc:66-109, 465-486)
    const bool own = lane < H;
    const int k = own ? lane : lane - H, p = own ? cur : other;
    if (k < st[O_HLEN + p]) {
      bit0 = (own ? 0 : L::o_hands) + k * L::BPC + st[hand_off(p, k)];
      v0 = 1u;
    }
  } else if (lane < 2 * H + P * H) {
    // card knowledge (canonical_encoders.cc:370-423): player rel (observer first), slot k
    const int idx = lane - 2 * H, rel = idx / H, k = idx - rel * H, p = (cur + rel) % P;
    if (k < st[O_HLEN + p]) {
      const int o = hand_off(p, k);
      const uint32_t cm = st[o + 1], rm = st[o + 2];
#pragma unroll
      for (int c = 0; c < C; ++c)
        if ((cm >> c) & 1u) v0 |= rm << (c * R);
      bit0 = L::o_know + idx * L::PER_CARD;
      if (st[o + 3] != kNone) v1 |= 1u << st[o + 3];
      if (st[o + 4] != kNone) v1 |= 1u << (C + st[o + 4]);
      bit1 = bit0 + L::BPC;
    }
  } else if (lane < 2 * H + P * H + C) {
    // discards of one colour: thermometers of widths 3,2,..,2,1 (canonical_encoders.cc:192-215)
    const int c = lane - 2 * H - P * H;
    v0 = ones(st[O_DISC + c * R]);
#pragma unroll
    for (int r = 1; r < R; ++r) v0 |= ones(st[O_DISC + c * R + r]) << (3 + 2 * (r - 1));
    bit0 = L::o_disc + c * L::PER_COLOR;
  } else if (lane == 2 * H + P * H + C) {
    // last non-deal move, observer-relative (canonical_encoders.cc:240-342)
    if (st[O_LMVALID]) {
      const int ty = st[O_LMTYPE];
      const bool reveal = ty == MV_REVEAL_COLOR || ty == MV_REVEAL_RANK, pd = ty == MV_PLAY || ty == MV_DISCARD;
      const int rel = (st[O_LMPLAYER] - cur + P) % P;
      v0 = 1u << rel;
      v0 |= 1u << (P + (ty == MV_PLAY ? 0 : ty == MV_DISCARD ? 1 : ty == MV_REVEAL_COLOR ? 2 : 3));
      if (reveal) v0 |= 1u << (P + 4 + (rel + st[O_LMTGT]) % P);
      if (ty == MV_REVEAL_COLOR) v0 |= 1u << (P + 4 + P + st[O_LMCOLOR]);
      if (ty == MV_REVEAL_RANK) v0 |= 1u << (P + 4 + P + C + st[O_LMRANK]);
      if (reveal) v0 |= (uint32_t)(st[O_LMREVEAL] & ((1 << H) - 1)) << (P + 4 + P + C + R);
      if (pd) v0 |= 1u << (P + 4 + P + C + R + H + st[O_LMIDX]);
      bit0 = L::o_last;
      if (pd) v1 |= 1u << st[O_LMCARD];
      if (ty == MV_PLAY) v1 |= (uint32_t)(st[O_LMFLAGS] & 3) << L::BPC;
      bit1 = L::o_last + L::LAST_A;
    }
  }
  // board fields: second field of the hand lanes (H = 2 leaves four hand lanes: they take two rounds)
  for (int f = lane; f < 7 && lane < 2 * H; f += 2 * H) {
    uint32_t v = 0;
    int bit = 0;
    const int n = st[O_DECK];
    if (f == 0) {          // fireworks: one-hot of (height - 1) per colour (canonical_encoders.cc:143-151)
#pragma unroll
      for (int c = 0; c < C; ++c)
        if (st[O_FW + c] > 0) v |= 1u << (c * R + st[O_FW + c] - 1);
      bit = L::o_fw;
    } else if (f == 1) {   // "hand is short" bits, observer first
      v = (st[O_HLEN + cur] < H ? 1u : 0u) | (st[O_HLEN + other] < H ? 2u : 0u);
      bit = L::o_miss;
    } else if (f == 2) {   // deck thermometer, first word
      v = ones(n < 32 ? n : 32);
      bit = L::o_deck;
    } else if (f == 3) {   // deck thermometer, second word
      v = n > 32 ? ones(n - 32) : 0u;
      bit = L::o_deck + 32;
    } else if (f == 4) {
      v = ones(st[O_INFO]);
      bit = L::o_info;
    } else if (f == 5) {
      v = ones(st[O_LIFE]);
      bit = L::o_life;
    } else {               // absolute current-player one-hot (rl_env.py:256-257)
      v = 1u << cur;
      bit = L::o_turn;
    }
    if (f < 2 * H) { v1 = v; bit1 = bit; }
    else or_bits(w, bit, v);          // only for H = 2 (second round of the four hand lanes)
  }
  or_bits(w, bit0, v0);
  or_bits(w, bit1, v1);
}

// bits [bit0, bit0 + n) of `words` (one spare word follows the last) as n bytes of 0/1; four bytes per lane
// and store when the row is 4-byte aligned, so a warp store covers 128 contiguous bytes
__device__ __forceinline__ void store_bits_u8(uint8_t* dst, const uint32_t* words, int bit0, int n, int lane) {
  if ((reinterpret_cast<uintptr_t>(dst) & 3u) == 0) {
    const int n4 = n >> 2;
    for (int g4 = lane; g4 < n4; g4 += HZ_WARP) {
      const int b = bit0 + 4 * g4;
      const uint32_t x = __funnelshift_r(words[b >> 5], words[(b >> 5) + 1], b & 31) & 15u;
      reinterpret_cast<uint32_t*>(dst)[g4] = (x & 1u) | ((x & 2u) << 7) | ((x & 4u) << 14) | ((x & 8u) << 21);
    }
    const int j = 4 * n4 + lane;
    if (j < n) dst[j] = (uint8_t)((words[(bit0 + j) >> 5] >> ((bit0 + j) & 31)) & 1u);
  } else {
    for (int j = lane; j < n; j += HZ_WARP) dst[j] = (uint8_t)((words[(bit0 + j) >> 5] >> ((bit0 + j) & 31)) & 1u);
  }
}

struct EnvView {
  uint8_t* state;   // [N][128]
  uint32_t* mt;     // [N][624]
  int32_t* mti;     // [N]
  int32_t* err;     // sticky: 1 + index of the first game that submitted an illegal move
  int N;
  Rules g;
};

struct EnvArgs {
  const uint8_t* reset_mask;
  const int32_t* actions;
  const uint8_t* active;
  int auto_reset;
  int32_t* out_reward;
  uint8_t* out_done;
  int32_t* out_score;
  float* out_global;
  int64_t ld_global;
  float* out_local;
  int64_t ld_local;
  float* out_legal;
  int32_t* out_dump;
  // byte-valued (0/1) observation outputs: the encoder's own value type (vector<int> of 0/1,
  // canonical_encoders.cc:441-486) at a quarter of the float traffic; strides shared with the float rows
  uint8_t* out_global8;
  uint8_t* out_local8;
  uint8_t* out_legal8;
  // bit-packed result row per game (hz_envs_step_observe_bits): the global observation as ceil(global_dim / 32)
  // little-endian words (bit j of the observation = word[j >> 5] >> (j & 31) & 1), then legal-move mask, reward,
  // done, score — everything a host-side caller needs from a step in one ~116-byte row
  uint32_t* out_bits;
  int64_t ld_bits;
  uint32_t* out_meta;   // optional [N][4]: {legal mask, reward, done, score} kept apart from the observation words
  // fused random policy (hz_envs_set_random_policy): every observing launch also draws a uniformly random legal move
  // of the position it observes — the k-th set bit of the legal mask, k from the splitmix64 finaliser over
  // (seed, game, draws made so far), bit-identical to hz_host_random_legal(.., seed, step = draws made so far)
  int32_t* policy_out;
  uint32_t* policy_ctr;
  unsigned long long policy_seed;
  // terminal rows (hz_envs_step_observe_u8_terminal, the TERM instantiation only): the observation of a finished game's
  // terminal state in the view of out_global8 / out_local8, and its legal mask, written before the re-deal
  uint8_t* out_term8;
  int64_t ld_term;
  uint8_t* out_term_legal8;
};

// TERM: the recording variant of step + auto-reset + byte observe; a separate instantiation, so the others carry none
// of its code
template <int C, int R, int H, int MI, int ML, bool RESET, bool STEP, bool OBSERVE, bool TERM = false>
__global__ void __launch_bounds__(kEnvWarps* HZ_WARP, 8) k_env(EnvView ev, EnvArgs a) {
  using L = ObsLayout<C, R, H, MI, ML>;
  __shared__ uint32_t s_state[kEnvWarps][kStateBytes / 4];
  __shared__ double s_scratch[kEnvWarps][64];
  __shared__ uint32_t s_obs[kEnvWarps][L::WORDS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gi = blockIdx.x * kEnvWarps + warp;
  if (gi >= ev.N) return;
  // the rules as compile-time constants (the helpers are force-inlined, so divisions by R, C fold away)
  const Rules g{C, R, H, MI, ML, 2 * H + (P - 1) * C + (P - 1) * R, L::ENC, L::OWN, L::DECK_MAX};
  uint8_t* st = reinterpret_cast<uint8_t*>(s_state[warp]);
  double* scratch = s_scratch[warp];
  uint32_t* gstate = reinterpret_cast<uint32_t*>(ev.state + (size_t)gi * kStateBytes);
  uint32_t* mt = ev.mt + (size_t)gi * 624;
  s_state[warp][lane] = gstate[lane];
  int mti = ev.mti[gi];
  const int mti0 = mti;
  MtWindow win = mt_prefetch(mt, mti, lane);
  __syncwarp();
  bool dirty = false;
  int reward = 0, done = 0, score = 0;
  bool stepped = false;
  HZ_ESTAMP(0);

  if (RESET && (a.reset_mask == nullptr || a.reset_mask[gi])) {  // rl_env.py:249-252
    new_state(st, g, lane);
    while ((int8_t)st[O_CUR] == -1) deal_random<C * R>(st, g, mt, mti, win, scratch, lane, gi);
    dirty = true;
  }
  if (STEP && (a.active == nullptr || a.active[gi])) {  // rl_env.py:413-438
    const int action = a.actions[gi];
    stepped = true;
    score = score_of(st, C);
    const unsigned lm = legal_mask(st, g, lane);
    if (action < 0 || action >= g.A || !((lm >> action) & 1u)) {  // reference: REQUIRE(MoveIsLegal) aborts the process
      if (lane == 0) atomicCAS(ev.err, 0, gi + 1);
      done = is_terminal(st, g);
    } else {
      const int last_score = score;
      HZ_ESTAMP(1);
      apply_move(st, g, action, lane);
      __syncwarp();
      HZ_ESTAMP(2);
      while ((int8_t)st[O_CUR] == -1) deal_random<C * R>(st, g, mt, mti, win, scratch, lane, gi);
      HZ_ESTAMP(3);
      score = score_of(st, C);
      reward = score - last_score;
      done = is_terminal(st, g);
      dirty = true;
      if (done && a.auto_reset) {
        if (TERM) {   // GameHistory.append takes the terminal observation (rl_env.py:426-434): encode it before the re-deal
          uint32_t* words = s_obs[warp];
          for (int i = lane; i < L::WORDS; i += HZ_WARP) words[i] = 0u;
          __syncwarp();
          obs_build<C, R, H, MI, ML>(st, (int8_t)st[O_CUR], words, lane);
          __syncwarp();
          if (a.out_term8) {
            uint8_t* ot = a.out_term8 + (size_t)gi * a.ld_term;
            if (a.out_global8) store_bits_u8(ot, words, 0, L::GLOBAL, lane);
            else store_bits_u8(ot, words, L::OWN, L::GLOBAL - L::OWN, lane);
          }
          const unsigned term_legal = legal_mask(st, g, lane);   // no terminal check: non-zero here, as in the reference
          if (a.out_term_legal8 && lane < g.A) a.out_term_legal8[(size_t)gi * g.A + lane] = (term_legal >> lane) & 1u;
          __syncwarp();   // the OBSERVE block below clears these words again
        }
        new_state(st, g, lane);
        while ((int8_t)st[O_CUR] == -1) deal_random<C * R>(st, g, mt, mti, win, scratch, lane, gi);
#ifdef HZ_TRACE
        if (g_env_trace && lane == 0) g_env_trace[(size_t)gi * 16 + 9] += 1;
#endif
      }
      HZ_ESTAMP(4);
    }
    if (lane == 0) {
      if (a.out_reward) a.out_reward[gi] = reward;
      if (a.out_done) a.out_done[gi] = (uint8_t)done;
      if (a.out_score) a.out_score[gi] = score;
    }
  }
  if (dirty) {
    __syncwarp();
    gstate[lane] = s_state[warp][lane];
    if (lane == 0 && mti != mti0) ev.mti[gi] = mti;
  }
  HZ_ESTAMP(5);
  if (OBSERVE) {
    constexpr int BPC = C * R;
    const int cur = (int8_t)st[O_CUR];
    uint32_t* words = s_obs[warp];
    for (int i = lane; i < L::WORDS; i += HZ_WARP) words[i] = 0u;
    __syncwarp();
    obs_build<C, R, H, MI, ML>(st, cur, words, lane);
    __syncwarp();
    HZ_ESTAMP(6);
    float* og = a.out_global ? a.out_global + (size_t)gi * a.ld_global : nullptr;
    float* ol = a.out_local ? a.out_local + (size_t)gi * a.ld_local : nullptr;
    if (og || ol) {
#pragma unroll 5
      for (int it = 0; it < (L::GLOBAL + 31) / 32; ++it) {
        const int j = it * 32 + lane;
        const float v = ((words[it] >> lane) & 1u) ? 1.0f : 0.0f;
        if (j < L::GLOBAL) {
          if (og) og[j] = v;
          if (ol && j >= L::OWN) ol[j - L::OWN] = v;
        }
      }
    }
    uint8_t* og8 = a.out_global8 ? a.out_global8 + (size_t)gi * a.ld_global : nullptr;
    uint8_t* ol8 = a.out_local8 ? a.out_local8 + (size_t)gi * a.ld_local : nullptr;
    if (og8) store_bits_u8(og8, words, 0, L::GLOBAL, lane);
    if (ol8) store_bits_u8(ol8, words, L::OWN, L::GLOBAL - L::OWN, lane);
    HZ_ESTAMP(7);
    if (a.out_legal || a.out_legal8 || a.out_bits || a.policy_out) {
      const unsigned legal_bits = legal_mask(st, g, lane);
      if (a.policy_out && lane == 0) {
        const uint32_t n = a.policy_ctr[gi];
        unsigned long long x = a.policy_seed + 0x9E3779B97F4A7C15ull * ((unsigned long long)gi + 1ull) + ((unsigned long long)n << 32);
        x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
        x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
        const uint32_t c = (uint32_t)__popc(legal_bits);
        const uint32_t k = (uint32_t)(((x >> 32) * c) >> 32);          // uniform in [0, popcount)
        a.policy_out[gi] = c ? (int32_t)(__fns(legal_bits, 0, (int)k + 1)) : 0;   // position of the k-th set bit
        a.policy_ctr[gi] = n + 1u;
      }
      if (lane < g.A) {
        const bool ok = (legal_bits >> lane) & 1u;
        if (a.out_legal) a.out_legal[(size_t)gi * g.A + lane] = ok ? 1.0f : 0.0f;
        if (a.out_legal8) a.out_legal8[(size_t)gi * g.A + lane] = ok ? 1 : 0;
      }
      if (a.out_bits) {
        constexpr int GW = (L::GLOBAL + 31) / 32;
        uint32_t* row = a.out_bits + (size_t)gi * a.ld_bits;
        if (lane < GW) row[lane] = words[lane];
        if (!stepped) {   // observe after reset: the episode's running score, nothing finished
          score = score_of(st, C);
          done = is_terminal(st, g);
        }
        if (lane == 0) {
          if (a.out_meta) {
            reinterpret_cast<uint4*>(a.out_meta)[gi] = make_uint4(legal_bits, (uint32_t)reward, (uint32_t)done, (uint32_t)score);
          } else {
            row[GW] = legal_bits;
            row[GW + 1] = (uint32_t)reward;
            row[GW + 2] = (uint32_t)done;
            row[GW + 3] = (uint32_t)score;
          }
        }
      }
    }
    HZ_ESTAMP(8);
    if (a.out_dump && lane == 0) {  // layout of oracle/hanabi_oracle.c:ohanabi_dump
      int32_t* o = a.out_dump + (size_t)gi * (5 + C + 2 * BPC + P * (1 + 5 * H));
      int n = 0;
      o[n++] = cur; o[n++] = st[O_INFO]; o[n++] = st[O_LIFE]; o[n++] = st[O_DECK];
      o[n++] = is_terminal(st, g);
      for (int c = 0; c < C; ++c) o[n++] = st[O_FW + c];
      for (int i = 0; i < BPC; ++i) o[n++] = st[O_DECKCNT + i];
      for (int i = 0; i < BPC; ++i) o[n++] = st[O_DISC + i];
      for (int p = 0; p < P; ++p) {
        o[n++] = st[O_HLEN + p];
        for (int k = 0; k < H; ++k) {
          const int ho = hand_off(p, k);
          if (k < st[O_HLEN + p]) {
            o[n++] = st[ho]; o[n++] = st[ho + 1]; o[n++] = st[ho + 2];
            o[n++] = (int8_t)st[ho + 3]; o[n++] = (int8_t)st[ho + 4];
          } else {
            o[n++] = -1; o[n++] = 0; o[n++] = 0; o[n++] = -1; o[n++] = -1;
          }
        }
      }
    }
  }
}

__global__ void k_mt_seed(uint32_t* mt, int32_t* mti, const int32_t* seeds, int N) {
  // std::mt19937::seed(value) (hanabi_game.cc:51): sequential recurrence, one thread per game
  const int gi = blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= N) return;
  uint32_t* m = mt + (size_t)gi * 624;
  uint32_t x = (uint32_t)seeds[gi];
  m[0] = x;
  for (int i = 1; i < 624; ++i) {
    x = 1812433253u * (x ^ (x >> 30)) + (uint32_t)i;
    m[i] = x;
  }
  mti[gi] = 624;
}

}  // namespace hz

using namespace hz;

struct hz_envs {
  int device = 0, N = 0, preset = 0;
  Rules g{};
  uint8_t* state = nullptr;
  uint32_t* mt = nullptr;
  int32_t* mti = nullptr;
  int32_t* err = nullptr;
  bool started = false;
  int dump_len = 0;
  cudaEvent_t host_done = nullptr;   // completion of the last hz_envs_host_step (created on first use)
  int32_t* policy_out = nullptr;     // fused random policy (hz_envs_set_random_policy): caller-owned dev int32[N]
  uint32_t* policy_ctr = nullptr;    // draws made per game (owned)
  unsigned long long policy_seed = 0;
  EnvView view() const { return EnvView{state, mt, mti, err, N, g}; }
};

template <bool RESET, bool STEP, bool OBSERVE, bool TERM = false>
static int launch_env(hz_envs* e, cudaStream_t s, const EnvArgs& args) {
  EnvArgs a = args;
  if (OBSERVE) { a.policy_out = e->policy_out; a.policy_ctr = e->policy_ctr; a.policy_seed = e->policy_seed; }
  dim3 grid((e->N + kEnvWarps - 1) / kEnvWarps), block(kEnvWarps * HZ_WARP);
  if (e->preset == 0) {
    k_env<5, 5, 5, 8, 3, RESET, STEP, OBSERVE, TERM><<<grid, block, 0, s>>>(e->view(), a);
  } else {
    k_env<2, 5, 2, 3, 1, RESET, STEP, OBSERVE, TERM><<<grid, block, 0, s>>>(e->view(), a);
  }
  HZ_LAUNCH_CHECK("k_env");
  return HZ_OK;
}

extern "C" {
#pragma GCC visibility push(default)

int hz_envs_create(hz_envs** out, int device, int num_games, int preset, const int32_t* seeds) {
  if (!out || num_games <= 0 || (preset != 0 && preset != 1) || !seeds) {
    set_error("hz_envs_create: need num_games>0, preset in {0,1}, host seeds[num_games]");
    return HZ_ERR_ARG;
  }
  DeviceGuard dg(device);
  if (!dg.ok) { set_error("hz_envs_create: cannot select device %d", device); return HZ_ERR_CUDA; }
  hz_envs* e = new hz_envs;
  e->device = device;
  e->N = num_games;
  e->preset = preset;
  Rules& g = e->g;
  if (preset == 0) { g.C = 5; g.R = 5; g.H = 5; g.max_info = 8; g.max_life = 3; }
  else { g.C = 2; g.R = 5; g.H = 2; g.max_info = 3; g.max_life = 1; }
  const int bpc = g.C * g.R, per_color = 3 + 2 * (g.R - 2) + 1;
  g.deck_max = per_color * g.C;
  g.A = 2 * g.H + (P - 1) * g.C + (P - 1) * g.R;
  g.own_len = g.H * bpc;
  g.enc_len = ((P - 1) * g.H * bpc + P) + (g.deck_max - P * g.H + bpc + g.max_info + g.max_life) +
              g.deck_max + (P + 4 + P + g.C + g.R + g.H + g.H + bpc + 2) + P * g.H * (bpc + g.C + g.R);
  e->dump_len = 5 + g.C + 2 * bpc + P * (1 + 5 * g.H);
  const size_t n = (size_t)num_games;
  int32_t* dseeds = nullptr;
  cudaError_t err = cudaSuccess;
  auto alloc = [&](void** p, size_t bytes) { if (err == cudaSuccess) err = cudaMalloc(p, bytes); };
  alloc((void**)&e->state, n * kStateBytes);
  alloc((void**)&e->mt, n * 624 * sizeof(uint32_t));
  alloc((void**)&e->mti, n * sizeof(int32_t));
  alloc((void**)&e->err, sizeof(int32_t));
  alloc((void**)&dseeds, n * sizeof(int32_t));
  if (err == cudaSuccess) err = cudaMemset(e->state, 0, n * kStateBytes);
  if (err == cudaSuccess) err = cudaMemset(e->err, 0, sizeof(int32_t));
  if (err == cudaSuccess) err = cudaMemcpy(dseeds, seeds, n * sizeof(int32_t), cudaMemcpyHostToDevice);
  if (err == cudaSuccess) {
    k_mt_seed<<<(num_games + 127) / 128, 128>>>(e->mt, e->mti, dseeds, num_games);
    g_launches.fetch_add(1);
    err = cudaDeviceSynchronize();
  }
  cudaFree(dseeds);
  if (err != cudaSuccess) {
    hz_envs_destroy(e);
    return fail_cuda(err, "hz_envs_create");
  }
  *out = e;
  return HZ_OK;
}

int hz_envs_destroy(hz_envs* e) {
  if (!e) return HZ_OK;
  DeviceGuard dg(e->device);
  cudaFree(e->state); cudaFree(e->mt); cudaFree(e->mti); cudaFree(e->err);
  if (e->host_done) cudaEventDestroy(e->host_done);
  cudaFree(e->policy_ctr);
  delete e;
  return HZ_OK;
}

int hz_envs_dims(const hz_envs* e, int32_t* out) {
  if (!e || !out) { set_error("hz_envs_dims: NULL argument"); return HZ_ERR_ARG; }
  const Rules& g = e->g;
  const int v[12] = {g.enc_len, g.own_len, P, g.A, g.C, g.R, g.H, g.max_info, g.max_life,
                     g.enc_len + P, g.own_len + g.enc_len + P, e->dump_len};
  for (int i = 0; i < 12; ++i) out[i] = v[i];
  return HZ_OK;
}

int hz_envs_reset(hz_envs* e, void* stream, const uint8_t* reset_mask) {
  if (!e) { set_error("hz_envs_reset: NULL handle"); return HZ_ERR_ARG; }
  DeviceGuard dg(e->device);
  EnvArgs a{};
  a.reset_mask = reset_mask;
  if (int rc = launch_env<true, false, false>(e, (cudaStream_t)stream, a)) return rc;
  e->started = true;
  return HZ_OK;
}

static int check_obs_args(const hz_envs* e, const void* og, int64_t ldg, const void* ol, int64_t ldl) {
  if ((og && ldg < e->g.own_len + e->g.enc_len + P) || (ol && ldl < e->g.enc_len + P)) {
    set_error("observation row stride smaller than the observation");
    return HZ_ERR_ARG;
  }
  return HZ_OK;
}

int hz_envs_step(hz_envs* e, void* stream, const int32_t* actions, const uint8_t* active,
                 int32_t* out_reward, uint8_t* out_done, int32_t* out_score) {
  if (!e || !actions) { set_error("hz_envs_step: NULL argument"); return HZ_ERR_ARG; }
  if (!e->started) { set_error("hz_envs_step: reset first"); return HZ_ERR_STATE; }
  DeviceGuard dg(e->device);
  EnvArgs a{};
  a.actions = actions; a.active = active;
  a.out_reward = out_reward; a.out_done = out_done; a.out_score = out_score;
  return launch_env<false, true, false>(e, (cudaStream_t)stream, a);
}

int hz_envs_observe(hz_envs* e, void* stream, float* out_global, int64_t ld_global,
                    float* out_local, int64_t ld_local, float* out_legal) {
  if (!e) { set_error("hz_envs_observe: NULL handle"); return HZ_ERR_ARG; }
  if (!e->started) { set_error("hz_envs_observe: reset first"); return HZ_ERR_STATE; }
  if (int rc = check_obs_args(e, out_global, ld_global, out_local, ld_local)) return rc;
  DeviceGuard dg(e->device);
  EnvArgs a{};
  a.out_global = out_global; a.ld_global = ld_global;
  a.out_local = out_local; a.ld_local = ld_local; a.out_legal = out_legal;
  return launch_env<false, false, true>(e, (cudaStream_t)stream, a);
}

int hz_envs_step_observe(hz_envs* e, void* stream, const int32_t* actions, const uint8_t* active,
                         int auto_reset, int32_t* out_reward, uint8_t* out_done, int32_t* out_score,
                         float* out_global, int64_t ld_global, float* out_local, int64_t ld_local,
                         float* out_legal) {
  if (!e || !actions) { set_error("hz_envs_step_observe: NULL argument"); return HZ_ERR_ARG; }
  if (!e->started) { set_error("hz_envs_step_observe: reset first"); return HZ_ERR_STATE; }
  if (int rc = check_obs_args(e, out_global, ld_global, out_local, ld_local)) return rc;
  DeviceGuard dg(e->device);
  EnvArgs a{};
  a.actions = actions; a.active = active; a.auto_reset = auto_reset;
  a.out_reward = out_reward; a.out_done = out_done; a.out_score = out_score;
  a.out_global = out_global; a.ld_global = ld_global;
  a.out_local = out_local; a.ld_local = ld_local; a.out_legal = out_legal;
  return launch_env<false, true, true>(e, (cudaStream_t)stream, a);
}

int hz_envs_observe_u8(hz_envs* e, void* stream, uint8_t* out_global, int64_t ld_global, uint8_t* out_local,
                       int64_t ld_local, uint8_t* out_legal) {
  if (!e) { set_error("hz_envs_observe_u8: NULL handle"); return HZ_ERR_ARG; }
  if (!e->started) { set_error("hz_envs_observe_u8: reset first"); return HZ_ERR_STATE; }
  if (int rc = check_obs_args(e, out_global, ld_global, out_local, ld_local)) return rc;
  DeviceGuard dg(e->device);
  EnvArgs a{};
  a.out_global8 = out_global; a.ld_global = ld_global;
  a.out_local8 = out_local; a.ld_local = ld_local; a.out_legal8 = out_legal;
  return launch_env<false, false, true>(e, (cudaStream_t)stream, a);
}

int hz_envs_step_observe_u8(hz_envs* e, void* stream, const int32_t* actions, const uint8_t* active,
                            int auto_reset, int32_t* out_reward, uint8_t* out_done, int32_t* out_score,
                            uint8_t* out_global, int64_t ld_global, uint8_t* out_local, int64_t ld_local,
                            uint8_t* out_legal) {
  if (!e || !actions) { set_error("hz_envs_step_observe_u8: NULL argument"); return HZ_ERR_ARG; }
  if (!e->started) { set_error("hz_envs_step_observe_u8: reset first"); return HZ_ERR_STATE; }
  if (int rc = check_obs_args(e, out_global, ld_global, out_local, ld_local)) return rc;
  DeviceGuard dg(e->device);
  EnvArgs a{};
  a.actions = actions; a.active = active; a.auto_reset = auto_reset;
  a.out_reward = out_reward; a.out_done = out_done; a.out_score = out_score;
  a.out_global8 = out_global; a.ld_global = ld_global;
  a.out_local8 = out_local; a.ld_local = ld_local; a.out_legal8 = out_legal;
  return launch_env<false, true, true>(e, (cudaStream_t)stream, a);
}

int hz_envs_step_observe_u8_terminal(hz_envs* e, void* stream, const int32_t* actions, const uint8_t* active,
                                     int32_t* out_reward, uint8_t* out_done, int32_t* out_score, uint8_t* out_global,
                                     int64_t ld_global, uint8_t* out_local, int64_t ld_local, uint8_t* out_legal,
                                     uint8_t* out_term, int64_t ld_term, uint8_t* out_term_legal) {
  if (!e || !actions) { set_error("hz_envs_step_observe_u8_terminal: NULL argument"); return HZ_ERR_ARG; }
  if (!e->started) { set_error("hz_envs_step_observe_u8_terminal: reset first"); return HZ_ERR_STATE; }
  if (!out_global == !out_local) {
    set_error("hz_envs_step_observe_u8_terminal: exactly one of out_global / out_local (the terminal rows' view)");
    return HZ_ERR_ARG;
  }
  if (int rc = check_obs_args(e, out_global, ld_global, out_local, ld_local)) return rc;
  const int width = out_global ? e->g.own_len + e->g.enc_len + P : e->g.enc_len + P;
  if (out_term && ld_term < width) {
    set_error("hz_envs_step_observe_u8_terminal: terminal row stride %lld smaller than the observation (%d)",
              (long long)ld_term, width);
    return HZ_ERR_ARG;
  }
  DeviceGuard dg(e->device);
  EnvArgs a{};
  a.actions = actions; a.active = active; a.auto_reset = 1;
  a.out_reward = out_reward; a.out_done = out_done; a.out_score = out_score;
  a.out_global8 = out_global; a.ld_global = ld_global;
  a.out_local8 = out_local; a.ld_local = ld_local; a.out_legal8 = out_legal;
  a.out_term8 = out_term; a.ld_term = ld_term; a.out_term_legal8 = out_term_legal;
  return launch_env<false, true, true, true>(e, (cudaStream_t)stream, a);
}

int hz_envs_step_observe_bits(hz_envs* e, void* stream, const int32_t* actions, const uint8_t* active, int auto_reset,
                              uint32_t* out_bits, int64_t ld_bits, uint32_t* out_meta) {
  if (!e || !out_bits) { set_error("hz_envs_step_observe_bits: NULL argument"); return HZ_ERR_ARG; }
  if (!e->started) { set_error("hz_envs_step_observe_bits: reset first"); return HZ_ERR_STATE; }
  const int gw = (e->g.own_len + e->g.enc_len + P + 31) / 32;
  const int need = gw + (out_meta ? 0 : 4);
  if (ld_bits < need) { set_error("hz_envs_step_observe_bits: rows need %d words", need); return HZ_ERR_ARG; }
  if (out_meta && ((uintptr_t)out_meta & 15)) { set_error("hz_envs_step_observe_bits: out_meta must be 16-byte aligned"); return HZ_ERR_ARG; }
  DeviceGuard dg(e->device);
  EnvArgs a{};
  a.actions = actions; a.active = active; a.auto_reset = auto_reset;
  a.out_bits = out_bits; a.ld_bits = ld_bits; a.out_meta = out_meta;
  if (actions) return launch_env<false, true, true>(e, (cudaStream_t)stream, a);
  return launch_env<false, false, true>(e, (cudaStream_t)stream, a);   // actions == NULL: observe only
}

// Host-facing step without staging copies.  Pinned (page-locked) host memory is device-addressable under unified
// addressing, so the kernel reads the actions from, and writes the packed rows to, the caller's host buffers itself:
// 116 bytes per game cross PCIe as posted writes from the SMs, and a step is ONE launch plus an event record instead
// of copy -> kernel -> copy -> copy.  hz_envs_host_wait blocks the calling host thread until that step's rows are in
// host memory (kernel completion flushes the writes).
int hz_envs_host_step(hz_envs* e, void* stream, const int32_t* h_actions, int auto_reset, uint32_t* h_bits,
                      int64_t ld_words, uint32_t* h_meta) {
  if (!e || !h_bits) { set_error("hz_envs_host_step: NULL argument"); return HZ_ERR_ARG; }
  DeviceGuard dg(e->device);
  const void* ptrs[3] = {h_actions, h_bits, h_meta};
  for (const void* p : ptrs) {
    if (!p) continue;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess || (at.type != cudaMemoryTypeHost && at.type != cudaMemoryTypeManaged &&
                                                            at.type != cudaMemoryTypeDevice)) {
      cudaGetLastError();
      set_error("hz_envs_host_step: buffers must be page-locked host memory (torch .pin_memory(), cudaHostAlloc)");
      return HZ_ERR_ARG;
    }
  }
  if (!e->host_done && cudaEventCreateWithFlags(&e->host_done, cudaEventDisableTiming) != cudaSuccess) {
    return fail_cuda(cudaGetLastError(), "hz_envs_host_step: event");
  }
  if (int rc = hz_envs_step_observe_bits(e, stream, h_actions, nullptr, auto_reset, h_bits, ld_words, h_meta)) return rc;
  const cudaError_t ce = cudaEventRecord(e->host_done, (cudaStream_t)stream);
  if (ce != cudaSuccess) return fail_cuda(ce, "hz_envs_host_step: record");
  return HZ_OK;
}

int hz_envs_set_random_policy(hz_envs* e, void* stream, int32_t* next_actions, uint64_t seed) {
  if (!e) { set_error("hz_envs_set_random_policy: NULL handle"); return HZ_ERR_ARG; }
  DeviceGuard dg(e->device);
  if (next_actions && !e->policy_ctr) {
    const cudaError_t ce = cudaMalloc(&e->policy_ctr, (size_t)e->N * sizeof(uint32_t));
    if (ce != cudaSuccess) return fail_cuda(ce, "hz_envs_set_random_policy: counters");
  }
  if (next_actions) HZ_CUDA(cudaMemsetAsync(e->policy_ctr, 0, (size_t)e->N * sizeof(uint32_t), (cudaStream_t)stream));
  e->policy_out = next_actions;
  e->policy_seed = seed;
  return HZ_OK;
}

int hz_envs_host_wait(hz_envs* e) {
  if (!e) { set_error("hz_envs_host_wait: NULL handle"); return HZ_ERR_ARG; }
  if (!e->host_done) return HZ_OK;   // nothing submitted yet
  const cudaError_t ce = cudaEventSynchronize(e->host_done);
  if (ce != cudaSuccess) return fail_cuda(ce, "hz_envs_host_wait");
  return HZ_OK;
}

// hz_host_random_legal (the host-side policy helper of this API) lives in hz_host.cpp: plain host C++.

#ifdef HZ_TRACE
int hz_debug_set_env_trace(long long* dev_buf) {   // debug build only (not in include/hzb200.h)
  return cudaMemcpyToSymbol(g_env_trace, &dev_buf, sizeof(dev_buf)) == cudaSuccess ? HZ_OK : HZ_ERR_CUDA;
}
#endif

int hz_envs_check(hz_envs* e, void* stream, int32_t* out_game) {
  if (!e) { set_error("hz_envs_check: NULL handle"); return HZ_ERR_ARG; }
  DeviceGuard dg(e->device);
  int32_t v = 0;
  HZ_CUDA(cudaMemcpyAsync(&v, e->err, sizeof(v), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  HZ_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  if (v != 0) {
    HZ_CUDA(cudaMemsetAsync(e->err, 0, sizeof(v), (cudaStream_t)stream));
    if (out_game) *out_game = v - 1;
    set_error("illegal Hanabi move submitted by game %d (the reference aborts here: "
              "REQUIRE(MoveIsLegal), hanabi_state.cc:222); the game was left untouched", v - 1);
    return HZ_ERR_ILLEGAL;
  }
  return HZ_OK;
}

int hz_envs_dump(hz_envs* e, void* stream, int32_t* out) {
  if (!e || !out) { set_error("hz_envs_dump: NULL argument"); return HZ_ERR_ARG; }
  if (!e->started) { set_error("hz_envs_dump: reset first"); return HZ_ERR_STATE; }
  DeviceGuard dg(e->device);
  EnvArgs a{};
  a.out_dump = out;
  return launch_env<false, false, true>(e, (cudaStream_t)stream, a);
}

#pragma GCC visibility pop
}  // extern "C"
