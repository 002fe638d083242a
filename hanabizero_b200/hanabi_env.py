"""Hanabi environment on the sm_100a game kernels.

`HanabiVecEnv` is the B200-native form: N independent games resident in HBM, stepped by one
kernel launch, observations / legal masks / rewards produced as CUDA tensors.

`HanabiEnv` is the drop-in for the reference's gym-like class
(/root/reference/envs/hanabi/rl_env.py:26-442): same constructor argument
(`{'hanabi_name': 'Hanabi-Full' | 'Hanabi-Small', 'seed': int | None}`), same `reset()` /
`step(action)` return tuples, same attributes the callers touch (`players`, `action_space[i].n`,
`num_moves()`, `vectorized_observation_shape()`, `vectorized_share_observation_shape()`, `game`,
`state`).  It is a one-game view of the same kernels — there is no Python or CPU game logic here.
"""
import numpy as np
import torch

from . import _lib
from ._lib import check, ptr

PRESETS = {"Hanabi-Full": 0, "Hanabi-Small": 1}  # rl_env.py:110-131
COLOR_CHAR = ["R", "Y", "G", "W", "B"]            # pyhanabi.py:26
CHANCE_PLAYER_ID = -1


class HanabiVecEnv:
    """N games of one preset on one GPU.  Game i owns its own std::mt19937 stream seeded with
    seeds[i], which persists across resets exactly like the reference's per-env HanabiGame object
    (rl_env.py:137,249)."""

    def __init__(self, num_games, hanabi_name="Hanabi-Full", seeds=None, device=None, obs_dtype=torch.float32):
        """obs_dtype: torch.float32 (what the network eats) or torch.uint8 (0/1 bytes: the encoder's own value
        type at a quarter of the traffic; rows are padded to a 16-byte multiple so the kernel stores words)."""
        if obs_dtype not in (torch.float32, torch.uint8):
            raise ValueError("obs_dtype must be torch.float32 or torch.uint8")
        self.obs_dtype = obs_dtype
        if hanabi_name not in PRESETS:
            raise ValueError("Unknown environment {}".format(hanabi_name))  # rl_env.py:133
        self.num_games = int(num_games)
        self.hanabi_name = hanabi_name
        from .cytree import _device_index   # device="cuda" (no index) means the CURRENT device, not cuda:0
        self.device_index = _device_index(device)
        self.device = torch.device("cuda", self.device_index)
        if seeds is None:
            seeds = np.zeros(self.num_games, np.int32)  # seed=None -> 0 (rl_env.py:106-109)
        seeds = np.ascontiguousarray(np.broadcast_to(np.asarray(seeds, np.int64), (self.num_games,)).astype(np.int32))
        self._lib = _lib.load()
        h = _lib.C.c_void_p()
        check(self._lib.hz_envs_create(_lib.C.byref(h), self.device_index, self.num_games,
                                       PRESETS[hanabi_name], seeds.ctypes.data))
        self._h = h
        dims = np.zeros(12, np.int32)
        check(self._lib.hz_envs_dims(self._h, dims.ctypes.data))
        (self.enc_len, self.own_len, self.players, self.num_actions, self.colors, self.ranks,
         self.hand_size, self.max_info, self.max_life, self.local_dim, self.global_dim,
         self.dump_len) = [int(x) for x in dims]
        n, dev = self.num_games, self.device
        self.reward = torch.zeros(n, dtype=torch.int32, device=dev)
        self.done = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.score = torch.zeros(n, dtype=torch.int32, device=dev)
        pad = (lambda d: (d + 15) // 16 * 16) if obs_dtype == torch.uint8 else (lambda d: d)
        self.global_obs = torch.zeros(n, pad(self.global_dim), dtype=obs_dtype, device=dev)[:, :self.global_dim]
        self.local_obs = torch.zeros(n, pad(self.local_dim), dtype=obs_dtype, device=dev)[:, :self.local_dim]
        self.legal = torch.zeros(n, self.num_actions, dtype=obs_dtype, device=dev)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None:
            try:
                self._lib.hz_envs_destroy(h)
            except Exception:
                pass
            self._h = None

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    @staticmethod
    def _ld(t):
        return 0 if t is None else t.stride(0)

    def reset_all(self, mask=None, observe=True):
        """HanabiEnv.reset for every game (or those with mask[i] != 0). Returns
        (global_obs, local_obs, legal) CUDA tensors when observe."""
        m = None if mask is None else mask.to(self.device, torch.uint8).contiguous()
        check(self._lib.hz_envs_reset(self._h, self._stream(), ptr(m)))
        if observe:
            return self.observe()

    def observe(self, out_global=None, out_local=None, out_legal=None, want_local=True, want_global=True):
        """Current player's observation tuple of every game, written into the given (possibly
        strided: row stride >= dim) float32 / uint8 CUDA tensors or the env's own buffers."""
        g = (self.global_obs if out_global is None else out_global) if want_global else None
        l = (self.local_obs if out_local is None else out_local) if want_local else None
        a = self.legal if out_legal is None else out_legal
        fn = self._lib.hz_envs_observe_u8 if self._all_u8(g, l, a) else self._lib.hz_envs_observe
        check(fn(self._h, self._stream(), ptr(g), self._ld(g), ptr(l), self._ld(l), ptr(a)))
        return g, l, a

    @staticmethod
    def _all_u8(*tensors):
        """True if the output tensors are uint8, False if float32; mixed sets are rejected."""
        kinds = {t.dtype for t in tensors if t is not None}
        if kinds <= {torch.uint8}:
            return bool(kinds)
        if kinds <= {torch.float32}:
            return False
        raise TypeError(f"observation outputs must be all float32 or all uint8, got {sorted(map(str, kinds))}")

    def step_all(self, actions, active=None, auto_reset=False, observe=True, out_global=None,
                 out_local=None, out_legal=None, want_local=True, want_global=True, out_terminal=None,
                 out_terminal_legal=None):
        """HanabiEnv.step for every (active) game in one launch.  actions: int32 CUDA tensor [N]
        (anything else is converted).  Returns (global_obs, local_obs, legal, reward, done, score).
        With auto_reset a finished game is re-dealt inside the same launch and the returned
        observation is the first one of its next episode (reward/done/score describe the finished
        step).  Illegal actions leave the game untouched; call check() to surface them.
        out_terminal / out_terminal_legal (uint8 CUDA [N, >= dim] / [N, A]; auto_reset=True, uint8 outputs and
        exactly one view only): a finished game's terminal observation, in that view, and its legal mask are written
        there before the re-deal (hz_envs_step_observe_u8_terminal); rows of the other games are left as they were."""
        terminal = out_terminal is not None or out_terminal_legal is not None
        if not (isinstance(actions, torch.Tensor) and actions.dtype == torch.int32 and actions.is_cuda):
            actions = torch.as_tensor(np.asarray(actions, np.int32) if not isinstance(actions, torch.Tensor)
                                      else actions, dtype=torch.int32).to(self.device)
        actions = actions.contiguous().view(-1)
        if actions.numel() != self.num_games:
            raise ValueError(f"expected {self.num_games} actions, got {actions.numel()}")
        act = None if active is None else active.to(self.device, torch.uint8).contiguous()
        if terminal and not (auto_reset and observe):
            raise ValueError("terminal rows need auto_reset=True and observe=True")
        if not observe:
            check(self._lib.hz_envs_step(self._h, self._stream(), ptr(actions), ptr(act),
                                         ptr(self.reward), ptr(self.done), ptr(self.score)))
            return None, None, None, self.reward, self.done, self.score
        g = (self.global_obs if out_global is None else out_global) if want_global else None
        l = (self.local_obs if out_local is None else out_local) if want_local else None
        a = self.legal if out_legal is None else out_legal
        if terminal:
            if not self._all_u8(g, l, a, out_terminal, out_terminal_legal):
                raise TypeError("terminal rows need uint8 observation, legal and terminal outputs")
            if (g is None) == (l is None):
                raise ValueError("terminal rows need exactly one observation view (want_global or want_local)")
            if out_terminal_legal is not None and (out_terminal_legal.shape != (self.num_games, self.num_actions)
                                                   or not out_terminal_legal.is_contiguous()):
                raise ValueError("out_terminal_legal must be a contiguous [num_games, num_actions] tensor")
            if out_terminal is not None and (out_terminal.dim() != 2 or out_terminal.shape[0] != self.num_games
                                             or out_terminal.stride(1) != 1):
                raise ValueError("out_terminal must be [num_games, >= dim] with unit column stride")
            check(self._lib.hz_envs_step_observe_u8_terminal(
                self._h, self._stream(), ptr(actions), ptr(act), ptr(self.reward), ptr(self.done), ptr(self.score),
                ptr(g), self._ld(g), ptr(l), self._ld(l), ptr(a), ptr(out_terminal), self._ld(out_terminal),
                ptr(out_terminal_legal)))
            return g, l, a, self.reward, self.done, self.score
        fn = self._lib.hz_envs_step_observe_u8 if self._all_u8(g, l, a) else self._lib.hz_envs_step_observe
        check(fn(self._h, self._stream(), ptr(actions), ptr(act), 1 if auto_reset else 0, ptr(self.reward),
                 ptr(self.done), ptr(self.score), ptr(g), self._ld(g), ptr(l), self._ld(l), ptr(a)))
        return g, l, a, self.reward, self.done, self.score

    # -- host-facing form: one bit-packed row per game -------------------------------------------------------------
    @property
    def bits_words(self):
        """Words per packed row: ceil(global_dim / 32) observation words + legal mask + reward + done + score."""
        return (self.global_dim + 31) // 32 + 4

    def step_bits(self, actions=None, active=None, auto_reset=False, out=None, out_meta=None):
        """One launch: step (actions int32 CUDA [N]; None = observe only) + optional auto-reset + the result of every
        game as ONE packed uint32 row (include/hzb200.h: hz_envs_step_observe_bits) — int32 CUDA tensor
        [N, bits_words], written into `out` if given.  ~116 bytes per Hanabi-Full game instead of 3.2 KB of float32.
        With `out_meta` (int32 CUDA [N, 4]) the four trailing words {legal mask, reward, done, score} go there and
        `out` may be [N, bits_words - 4]."""
        if out is None:
            out = torch.empty(self.num_games, self.bits_words - (0 if out_meta is None else 4), dtype=torch.int32,
                              device=self.device)
        act = None if active is None else active.to(self.device, torch.uint8).contiguous()
        check(self._lib.hz_envs_step_observe_bits(self._h, self._stream(), ptr(actions), ptr(act), 1 if auto_reset else 0,
                                                  ptr(out), out.stride(0), ptr(out_meta)))
        return out

    def unpack_bits(self, packed, meta=None):
        """Packed rows on the HOST (numpy int32/uint32 [n, bits_words] or a CPU tensor; or observation words [n, W] plus
        `meta` [n, 4]) -> dict of numpy arrays: global_obs uint8 [n, global_dim], local_obs uint8 [n, local_dim] (its
        suffix), legal uint8 [n, A], reward int32 [n], done bool [n], score int32 [n]."""
        as_u32 = lambda x: np.ascontiguousarray(x.numpy() if isinstance(x, torch.Tensor) else x).view(np.uint32)
        rows = as_u32(packed)
        w = self.bits_words - 4
        m = rows[:, w:w + 4] if meta is None else as_u32(meta)
        bits = np.unpackbits(np.ascontiguousarray(rows[:, :w]).view(np.uint8), axis=1, bitorder="little")[:, :self.global_dim]
        legal = (m[:, 0, None] >> np.arange(self.num_actions, dtype=np.uint32)) & 1
        return dict(global_obs=bits, local_obs=bits[:, self.own_len:], legal=legal.astype(np.uint8),
                    reward=np.ascontiguousarray(m[:, 1]).view(np.int32), done=m[:, 2] != 0,
                    score=np.ascontiguousarray(m[:, 3]).view(np.int32))

    def set_random_policy(self, next_actions, seed=0):
        """Fused random policy (hz_envs_set_random_policy): from now on every observing launch also writes a uniformly
        random legal move of each observed position into `next_actions` (int32 CUDA [N]; None switches it off) — hand
        the same tensor to the next step_all / step_bits and a random-play step is one kernel launch.  Draw d of game
        i equals random_legal_host(..., seed, step=d)[i]."""
        if next_actions is not None and (next_actions.dtype != torch.int32 or next_actions.numel() != self.num_games
                                         or not next_actions.is_cuda or not next_actions.is_contiguous()):
            raise ValueError("next_actions must be a contiguous int32 CUDA tensor with one entry per game")
        self._policy_buf = next_actions       # kept alive: the kernel writes into it
        check(self._lib.hz_envs_set_random_policy(self._h, self._stream(), ptr(next_actions), int(seed) & (2 ** 64 - 1)))

    def random_legal_host(self, rows, out_actions, seed=0, step=0):
        """HOST: a uniformly random legal move per game into `out_actions` (CPU int32 tensor [n], e.g. pinned) from
        host rows holding the legal-mask word: packed rows [n, bits_words] (word W) or meta rows [n, 4] (word 0) —
        hz_host_random_legal."""
        word = 0 if rows.shape[1] == 4 else self.bits_words - 4
        check(self._lib.hz_host_random_legal(rows.data_ptr(), rows.stride(0), word, rows.shape[0], self.num_actions,
                                             int(seed) & (2 ** 64 - 1), int(step) & 0xffffffff, out_actions.data_ptr()))
        return out_actions

    def check(self):
        """Synchronises and raises IllegalMoveError if any game was handed an illegal move."""
        bad = _lib.C.c_int32(-1)
        check(self._lib.hz_envs_check(self._h, self._stream(), _lib.C.byref(bad)))

    def dump(self):
        """int32 [N, dump_len] full hidden state (layout of oracle/hanabi_oracle.c:ohanabi_dump)."""
        out = torch.empty(self.num_games, self.dump_len, dtype=torch.int32, device=self.device)
        check(self._lib.hz_envs_dump(self._h, self._stream(), ptr(out)))
        return out


def frame_layout(hanabi_name, mdp, device=None):
    """(frame_dim, frame_words, bit_offset) of the observation frame a network of `hanabi_name` takes for `mdp`
    ("global" or "local"), read from the game kernels' own dimensions (hz_envs_dims): the frame is bits
    [bit_offset, bit_offset + frame_dim) of the packed string of frame_words words that step_bits / EnvPipeline(fmt="bits")
    hand out per game — the whole string for "global", its local suffix for "local"."""
    if mdp not in ("global", "local"):
        raise ValueError("mdp must be 'global' or 'local'")
    env = HanabiVecEnv(1, hanabi_name, device=device)
    words = (env.global_dim + 31) // 32
    if mdp == "global":
        return env.global_dim, words, 0
    return env.local_dim, words, env.global_dim - env.local_dim


class EnvPipeline:
    """Host-driven stepping, double-buffered like mcts.SearchPipeline: the games are held as several independent
    GROUPS (one HanabiVecEnv each); every group has its own stream on which a step is

        actions from pinned host memory -> one kernel (step + auto-reset + observe) -> result to pinned host memory

    so while the host reads one group's result and chooses its next actions, the other groups' copies and kernels are
    in flight.  A closed loop over a single batch cannot overlap anything (the next actions depend on the result);
    two half-batches can.

        pipe = EnvPipeline([env_a, env_b], fmt="bits")
        for g in range(pipe.groups): pipe.observe_now(g)
        while True:
            for g in range(pipe.groups):
                rows, legal = pipe.wait(g)               # pinned host tensors of group g's last step
                pipe.step(g, choose(rows, legal))        # pinned int32 [n_g]; returns at once

    fmt: "bits" = packed (HanabiVecEnv.step_bits / unpack_bits; `wait` returns (observation words int32 [n, W],
    meta int32 [n, 4] = {legal mask, reward, done, score})); "u8" / "f32" = (global observation [n, D], legal [n, A])
    as 0/1 bytes or float32 — what round 1 shipped, kept for comparison (8x / 32x the bytes).

    zero_copy (fmt="bits" only, default): no staging copies at all — the kernel reads the actions from and writes the
    packed rows to the pinned host buffers itself (hz_envs_host_step: one launch + one event record per step, two
    ctypes calls and no torch call on the host side of a step)."""

    def __init__(self, envs, fmt="bits", use_graphs=True, zero_copy=None):
        if fmt not in ("bits", "u8", "f32"):
            raise ValueError("fmt must be 'bits', 'u8' or 'f32'")
        self.envs = list(envs) if isinstance(envs, (list, tuple)) else [envs]
        self.fmt, self.groups, self.use_graphs = fmt, len(self.envs), bool(use_graphs)
        self.zero_copy = (fmt == "bits") if zero_copy is None else bool(zero_copy)
        if self.zero_copy and fmt != "bits":
            raise ValueError("zero_copy needs fmt='bits'")
        self.slots = []
        self.d2h_bytes_per_step = 0
        for env in self.envs:
            n, a, dev = env.num_games, env.num_actions, env.device
            if fmt == "bits":      # observation words and the four meta words {legal mask, reward, done, score} apart
                d_obs = torch.zeros(n, env.bits_words - 4, dtype=torch.int32, device=dev)
                d_leg = torch.zeros(n, 4, dtype=torch.int32, device=dev)
            else:
                dt = torch.uint8 if fmt == "u8" else torch.float32
                pad = (env.global_dim + 15) // 16 * 16 if fmt == "u8" else env.global_dim
                d_obs = torch.zeros(n, pad, dtype=dt, device=dev)
                d_leg = torch.zeros(n, a, dtype=dt, device=dev)
            h_obs = torch.empty(d_obs.shape, dtype=d_obs.dtype).pin_memory()
            h_leg = None if d_leg is None else torch.empty(d_leg.shape, dtype=d_leg.dtype).pin_memory()
            self.slots.append(dict(env=env, stream=torch.cuda.Stream(dev), d_act=torch.zeros(n, dtype=torch.int32, device=dev),
                                   h_act=torch.zeros(n, dtype=torch.int32).pin_memory(), graph=None, steps=0,
                                   d_obs=d_obs, d_leg=d_leg, h_obs=h_obs, h_leg=h_leg, done=torch.cuda.Event()))
            self.d2h_bytes_per_step += h_obs.numel() * h_obs.element_size() + (
                0 if h_leg is None else h_leg.numel() * h_leg.element_size())
            # everything enqueued on the creating stream so far (reset, ...) precedes the group's own stream
            self.slots[-1]["stream"].wait_stream(torch.cuda.current_stream(dev))

    def actions(self, group):
        """The group's pinned action buffer (int32 [n]): fill it in place and call step(group) to skip one host copy."""
        return self.slots[group]["h_act"]

    def _enqueue(self, s, with_actions):
        """actions in -> kernel -> results out, on the current stream (eager, or under graph capture)."""
        env = s["env"]
        acts = None
        if with_actions:
            acts = s["d_act"]
            acts.copy_(s["h_act"], non_blocking=True)
        if self.fmt == "bits":
            env.step_bits(acts, auto_reset=True, out=s["d_obs"], out_meta=s["d_leg"])
        elif acts is None:
            env.observe(out_global=s["d_obs"][:, :env.global_dim], out_legal=s["d_leg"], want_local=False)
        else:
            env.step_all(acts, auto_reset=True, want_local=False, out_global=s["d_obs"][:, :env.global_dim],
                         out_legal=s["d_leg"])
        s["h_obs"].copy_(s["d_obs"], non_blocking=True)
        if s["h_leg"] is not None:
            s["h_leg"].copy_(s["d_leg"], non_blocking=True)

    def _host_step(self, s, with_actions):
        env = s["env"]
        check(env._lib.hz_envs_host_step(env._h, s["stream"].cuda_stream, s["h_act"].data_ptr() if with_actions else None, 1,
                                         s["h_obs"].data_ptr(), s["h_obs"].stride(0), s["h_leg"].data_ptr()))

    def observe_now(self, group):
        """Current observation of the group's games (no step)."""
        s = self.slots[group]
        if self.zero_copy:
            return self._host_step(s, False)
        with torch.cuda.stream(s["stream"]):
            self._enqueue(s, False)
            s["done"].record(s["stream"])

    def step(self, group, h_actions=None):
        """Step the group's games with the given actions (host int32 [n]; None = the buffer from `actions(group)` was
        filled in place); returns at once.  After two eager steps the group's four operations (actions in, kernel,
        observation out, meta out) are captured once and replayed as one CUDA graph launch: the host-side cost of a
        step is what bounds a host-driven loop."""
        s = self.slots[group]
        if h_actions is not None and h_actions.data_ptr() != s["h_act"].data_ptr():
            s["h_act"].copy_(h_actions)
        if self.zero_copy:
            s["steps"] += 1
            return self._host_step(s, True)
        with torch.cuda.stream(s["stream"]):
            if s["graph"] is None and s["steps"] >= 2 and self.use_graphs:
                s["stream"].synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=s["stream"]):
                    self._enqueue(s, True)
                s["graph"] = g
                # the capture only recorded the step: it has not run yet
            if s["graph"] is not None:
                s["graph"].replay()
            else:
                self._enqueue(s, True)
            s["done"].record(s["stream"])
        s["steps"] += 1

    def wait(self, group):
        """Block until the group's last submission is in host memory; returns (observation rows, legal) host tensors —
        for fmt="bits": (observation words [n, W] int32, meta [n, 4] int32 = {legal mask, reward, done, score})."""
        s = self.slots[group]
        if self.zero_copy:
            check(s["env"]._lib.hz_envs_host_wait(s["env"]._h))
        else:
            s["done"].synchronize()
        return s["h_obs"], s["h_leg"]

    def drain(self):
        for s in self.slots:
            if self.zero_copy:
                check(s["env"]._lib.hz_envs_host_wait(s["env"]._h))
            else:
                s["done"].synchronize()
            torch.cuda.current_stream(s["env"].device).wait_stream(s["stream"])


class Discrete:
    """gym.spaces.Discrete stand-in (rl_env.py:21,141): the callers only read `.n`."""

    def __init__(self, n):
        self.n = n


class _GameView:
    """The part of pyhanabi.HanabiGame the env's callers use (pyhanabi.py:679-785)."""

    def __init__(self, vec):
        self._v = vec

    def num_players(self): return self._v.players
    def num_colors(self): return self._v.colors
    def num_ranks(self): return self._v.ranks
    def hand_size(self): return self._v.hand_size
    def max_information_tokens(self): return self._v.max_info
    def max_life_tokens(self): return self._v.max_life
    def max_moves(self): return self._v.num_actions

    def num_cards(self, color, rank):
        return 3 if rank == 0 else (1 if rank == self._v.ranks - 1 else 2)

    def get_move(self, move_uid):
        return move_dict(self._v, int(move_uid))

    def get_move_uid(self, move):
        return move_uid(self._v, move)


class _StateView:
    """Read-only view of pyhanabi.HanabiState (pyhanabi.py:495-660) decoded from the device state."""

    def __init__(self, vec):
        self._v = vec

    def _d(self):
        return self._v.dump()[0].cpu().numpy()

    def cur_player(self): return int(self._d()[0])
    def information_tokens(self): return int(self._d()[1])
    def life_tokens(self): return int(self._d()[2])
    def deck_size(self): return int(self._d()[3])
    def is_terminal(self): return bool(self._d()[4])
    def fireworks(self): return [int(x) for x in self._d()[5:5 + self._v.colors]]

    def score(self):
        d = self._d()
        return 0 if d[2] <= 0 else int(d[5:5 + self._v.colors].sum())

    def player_hands(self):
        v, d = self._v, self._d()
        base = 5 + v.colors + 2 * v.colors * v.ranks
        hands = []
        for p in range(v.players):
            off = base + p * (1 + 5 * v.hand_size)
            hands.append([{"color": COLOR_CHAR[int(d[off + 1 + 5 * k]) // v.ranks],
                           "rank": int(d[off + 1 + 5 * k]) % v.ranks} for k in range(int(d[off]))])
        return hands

    def discard_counts(self):
        v, d = self._v, self._d()
        o = 5 + v.colors + v.colors * v.ranks
        return d[o:o + v.colors * v.ranks].reshape(v.colors, v.ranks).tolist()


def move_dict(v, uid):
    """HanabiGame::ConstructMove (hanabi_game.cc:159-183) as the dict form of pyhanabi's to_dict."""
    h, c = v.hand_size, v.colors
    if uid < 0 or uid >= v.num_actions:
        raise ValueError(f"move uid {uid} out of range")
    if uid < h:
        return {"action_type": "DISCARD", "card_index": uid}
    if uid < 2 * h:
        return {"action_type": "PLAY", "card_index": uid - h}
    uid -= 2 * h
    if uid < (v.players - 1) * c:
        return {"action_type": "REVEAL_COLOR", "target_offset": 1 + uid // c, "color": COLOR_CHAR[uid % c]}
    uid -= (v.players - 1) * c
    return {"action_type": "REVEAL_RANK", "target_offset": 1 + uid // v.ranks, "rank": uid % v.ranks}


def move_uid(v, action):
    """HanabiGame::GetMoveUid (hanabi_game.cc:79-95) from the dict form (rl_env.py:516-575)."""
    assert isinstance(action, dict), "Expected dict, got: {}".format(action)
    assert "action_type" in action, "Action should contain `action_type`. action: {}".format(action)
    t, h = action["action_type"], v.hand_size
    if t == "DISCARD":
        return int(action["card_index"])
    if t == "PLAY":
        return h + int(action["card_index"])
    if t == "REVEAL_COLOR":
        assert isinstance(action["color"], str)
        return 2 * h + (int(action["target_offset"]) - 1) * v.colors + COLOR_CHAR.index(action["color"])
    if t == "REVEAL_RANK":
        return (2 * h + (v.players - 1) * v.colors + (int(action["target_offset"]) - 1) * v.ranks
                + int(action["rank"]))
    raise ValueError("Unknown action_type: {}".format(t))


class HanabiEnv:
    """Drop-in for envs.hanabi.rl_env.HanabiEnv (rl_env.py:26-442) backed by a one-game batch."""

    def __init__(self, args, device=None):
        seed = 0 if args["seed"] is None else args["seed"]  # rl_env.py:106-109
        self._vec = HanabiVecEnv(1, args["hanabi_name"], [seed], device=device, obs_dtype=torch.uint8)
        v = self._vec
        self.game = _GameView(v)
        self.state = None
        self.players = v.players
        self.action_space = [Discrete(v.num_actions) for _ in range(v.players)]
        self.observation_space = [[v.enc_len + v.players] for _ in range(v.players)]
        self.share_observation_space = [[v.own_len + v.enc_len + v.players] for _ in range(v.players)]
        self._action = torch.zeros(1, dtype=torch.int32, device=v.device)
        # one step = action in (4 bytes, pinned) -> one launch -> one packed row out (pinned) -> one synchronise
        self._h_action = torch.zeros(1, dtype=torch.int32).pin_memory()
        self._d_row = torch.zeros(1, v.bits_words, dtype=torch.int32, device=v.device)
        self._h_row = torch.zeros(1, v.bits_words, dtype=torch.int32).pin_memory()

    def vectorized_observation_shape(self):
        return [self._vec.enc_len]

    def vectorized_share_observation_shape(self):
        return [self._vec.own_len + self._vec.enc_len]

    def num_moves(self):
        return self._vec.num_actions

    def _fetch(self):
        """Packed row -> host -> the reference's Python lists (rl_env.py:254-263, 426-442)."""
        self._h_row.copy_(self._d_row, non_blocking=True)
        torch.cuda.current_stream(self._vec.device).synchronize()
        u = self._vec.unpack_bits(self._h_row)
        share_obs = u["global_obs"][0].astype(np.int64).tolist()
        obs = u["local_obs"][0].astype(np.int64).tolist()
        legal = list(u["legal"][0].astype(np.float64))
        return share_obs, obs, legal, int(u["reward"][0]), bool(u["done"][0]), int(u["score"][0])

    def reset(self, choose=True):
        """rl_env.py:148-267 -> (share_obs, obs, available_actions)."""
        if not choose:
            # the reference's choose=False branch references undefined names and cannot run
            raise NotImplementedError("reset(choose=False) is broken in the reference (rl_env.py:264-266)")
        self._vec.reset_all(observe=False)
        self._vec.step_bits(None, out=self._d_row)
        self.state = _StateView(self._vec)
        share_obs, obs, legal = self._fetch()[:3]
        self._legal_now = legal      # host copy of the mask: an illegal action is caught before it reaches the device
        return share_obs, obs, legal

    def step(self, action):
        """rl_env.py:292-442 -> (share_obs, obs, reward, done, {'score'}, available_actions)."""
        if isinstance(action, dict):
            uid = move_uid(self._vec, action)
        elif isinstance(action, int) and not isinstance(action, bool):
            assert action != -1  # rl_env.py:404-411 ends in `assert False`
            uid = action
        else:
            raise ValueError("Expected action as dict or int, got: {}".format(action))  # rl_env.py:415
        if self.state is None:
            raise RuntimeError("step() before reset()")
        if not self._legal_now[uid] if 0 <= uid < len(self._legal_now) else True:
            # the reference aborts the process here (REQUIRE(MoveIsLegal), hanabi_state.cc:222); the kernel leaves the
            # game untouched and flags it, which check() turns into the exception
            self._action.fill_(uid)
            self._vec.step_all(self._action, observe=False)
            try:
                self._vec.check()
            except _lib.IllegalMoveError as e:
                if isinstance(action, dict):  # rl_env.py:569-572
                    raise AssertionError("Illegal action: {}".format(action)) from e
                raise
        self._h_action[0] = uid
        self._action.copy_(self._h_action, non_blocking=True)
        self._vec.step_bits(self._action, out=self._d_row)
        share_obs, obs, legal, reward, done, score = self._fetch()
        self._legal_now = legal
        return share_obs, obs, reward, done, {"score": score}, legal

    def close(self):
        pass
