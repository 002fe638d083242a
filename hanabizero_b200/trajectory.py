"""Trajectory recording for N self-play games on the device — SURVEY.md §8f row N3.

The reference keeps one `GameHistory` per env in Python lists (/root/reference/core/game.py:49-215):
`init` (first frame replicated `stacked_observations` times + first legal mask, :73-93),
`store_search_stats` (root child visit distribution + root value, :189-204) and `append` (action, next
observation, reward, next legal mask, :143-148) per move, `game_over` (:176-187) at the end, and the
self-play worker reshapes rewards into "turn rewards" when it files the episode
(/root/reference/core/selfplay_worker.py:29-39).  Here the same record lives in HBM for all games
(`hz_traj_*`, include/hzb200.h): the env / search / sampler kernels' outputs are appended without leaving
the device, and only finished episodes cross to the host, already in `GameHistory.save_file`'s layout
(game.py:136-140).
"""
import numpy as np
import torch

from . import _lib
from ._lib import check, ptr


class TrajectoryOverflow(RuntimeError):
    pass


class TrajectoryRecorder:
    """`banks` record banks per game, used round-robin: up to banks - 1 finished episodes of a game can wait
    for `flush()` while the game plays on (call `flush()` at least every banks - 1 episodes of any game)."""

    def __init__(self, num_games, obs_dim, num_actions, stack=4, max_len=128, device=None, banks=2):
        self.n, self.obs_dim, self.actions = int(num_games), int(obs_dim), int(num_actions)
        self.stack, self.max_len, self.banks = int(stack), int(max_len), int(banks)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        n, dev, nb = self.n, self.device, self.banks
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
        self.obs = z((n, nb, self.stack + self.max_len, self.obs_dim), torch.uint8)
        self.legal = z((n, nb, self.max_len + 1, self.actions), torch.uint8)
        self.action = z((n, nb, self.max_len), torch.int32)
        self.reward = z((n, nb, self.max_len), torch.int32)
        self.visits = z((n, nb, self.max_len, self.actions), torch.int32)
        self.root_value = z((n, nb, self.max_len), torch.float32)
        self.len = z((n, nb), torch.int32)
        self.bank = z((n,), torch.uint8)
        self.finished = z((n, nb), torch.uint8)
        self.overflow = z((1,), torch.int32)
        self._lib = _lib.load()
        v = _lib.TrajView()
        for name in ("obs", "legal", "action", "reward", "visits", "root_value", "len", "bank", "finished", "overflow"):
            setattr(v, name, ptr(getattr(self, name)))
        v.num, v.obs_dim, v.actions, v.stack, v.max_len, v.banks = n, self.obs_dim, self.actions, self.stack, self.max_len, nb
        self._view = v
        self._ref = _lib.C.byref(v)

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    @staticmethod
    def _f32(t):
        if t.dtype != torch.float32 or not t.is_cuda:
            raise TypeError("observations and legal masks must be float32 CUDA tensors")
        return t

    def begin(self, obs, legal, mask=None):
        """GameHistory.init for the games with mask[i] != 0 (all if None).  obs float32 [N, >= obs_dim] (row
        stride free), legal float32 [N, A], mask uint8 [N]; CUDA."""
        obs, legal = self._f32(obs), self._f32(legal).contiguous()
        check(self._lib.hz_traj_begin(self._stream(), self._ref, ptr(obs), obs.stride(0), ptr(legal), ptr(mask)))

    def append(self, actions, obs, legal, reward, visits, root_values, done, active=None):
        """store_search_stats + append for one move of every (active) game; done closes the episode."""
        obs, legal = self._f32(obs), self._f32(legal).contiguous()
        check(self._lib.hz_traj_append(self._stream(), self._ref, ptr(actions), ptr(obs), obs.stride(0), ptr(legal),
                                       ptr(reward), ptr(visits), ptr(root_values), ptr(done), ptr(active)))

    def record_u8(self, actions, reward, visits, root_values, done, next_obs, next_legal, term_obs, term_legal,
                  active=None):
        """append + begin(mask=done) for one move of every game in one launch (hz_traj_record_u8), from uint8 rows:
        a finished game appends term_obs / term_legal (its terminal rows) and begins its next episode from next_obs /
        next_legal; the others append next_obs / next_legal.  Observation rows [N, >= obs_dim] (row stride free),
        legal rows [N, A]; CUDA."""
        for t in (next_obs, next_legal, term_obs, term_legal):
            if t.dtype != torch.uint8 or not t.is_cuda or t.stride(-1) != 1:
                raise TypeError("record_u8 takes uint8 CUDA rows with unit column stride")
        for t in (next_legal, term_legal):
            if t.stride(0) != self.actions:
                raise ValueError("legal rows must be [N, num_actions] contiguous")
        check(self._lib.hz_traj_record_u8(self._stream(), self._ref, ptr(actions), ptr(reward), ptr(visits),
                                          ptr(root_values), ptr(done), ptr(next_obs), next_obs.stride(0), ptr(next_legal),
                                          ptr(term_obs), term_obs.stride(0), ptr(term_legal), ptr(active)))

    def check(self):
        """Synchronises; raises if a game ran out of room since the last check."""
        bad = int(self.overflow.item())
        if bad:
            self.overflow.zero_()
            raise TrajectoryOverflow(f"game {bad - 1}: episode longer than max_len={self.max_len} or all banks "
                                     "full (flush() was not called in time); its record is incomplete")

    def flush(self, store=None):
        """Hand the finished episodes to the host.  Returns a list of dicts, one per episode, in the layout of
        GameHistory.save_file (game.py:136-140) after SelfPlay `put` (selfplay_worker.py:29-39):
          'game' int, 'vis' float64 [T, A], 'root' float64 [T], 'a' int64 [T], 'o' uint8 [stack + T, D],
          'r' int64 [T] turn rewards, 'r_raw' int64 [T] env rewards, 'la' float64 [T + 1, A].
        One small D2H (flags + lengths), one pack kernel, one D2H of the packed episodes.
        With `store` (an EpisodeStore of this recorder's obs_dim, num_actions, stack and device) the pack writes the
        frames and legal rows straight into the store's arenas, on the current stream, and each dict carries the
        episode's store id 'id' (int) in place of 'o'; the frames never cross to the host."""
        if store is not None:
            store._check_recorder(self)
        self.check()
        lens = torch.where(self.finished.bool(), self.len, torch.full_like(self.len, -1)).cpu().numpy()
        games, banks = np.nonzero(lens >= 0)
        if games.size == 0:
            return []
        # oldest first within a game: banks are filled round-robin and the bank being written comes last
        cur = self.bank.cpu().numpy().astype(np.int64)
        order = np.lexsort(((banks - cur[games] - 1) % self.banks, games))
        games, banks = games[order], banks[order]
        T = lens[games, banks].astype(np.int64)
        off = np.concatenate(([0], np.cumsum(T)[:-1])).astype(np.int64)
        total, E, dev = int(T.sum()), int(games.size), self.device
        idx = torch.from_numpy(np.stack((games.astype(np.int32), banks.astype(np.int32)))).to(dev)
        d_off = torch.from_numpy(off).to(dev)
        if store is None:
            o = torch.empty(total + E * self.stack, self.obs_dim, dtype=torch.uint8, device=dev)
            la = torch.empty(total + E, self.actions, dtype=torch.uint8, device=dev)
        else:       # the block's rows of the arenas, in the layout the pack writes
            ids, base = store._begin_add(T)
            o = store.frames[base:base + total + E * self.stack]
            la = store.legal[base:base + total + E]
        a = torch.empty(total, dtype=torch.int32, device=dev)
        r = torch.empty(total, dtype=torch.int32, device=dev)
        vis = torch.empty(total, self.actions, dtype=torch.int32, device=dev)
        root = torch.empty(total, dtype=torch.float32, device=dev)
        check(self._lib.hz_traj_pack(self._stream(), self._ref, E, ptr(idx[0]), ptr(idx[1]), ptr(d_off), ptr(o),
                                     ptr(la), ptr(a), ptr(r), ptr(vis), ptr(root)))
        if store is not None:
            store._end_add()
        pol = torch.empty(total, self.actions, dtype=torch.float64, device=dev)
        if total:
            check(self._lib.hz_visit_policy(self._stream(), ptr(vis), None, total, self.actions, ptr(pol), None))
        la, a, r, pol, root = (x.cpu().numpy() for x in (la, a, r, pol, root))
        o = o.cpu().numpy() if store is None else None
        out = []
        for e in range(E):
            s, t = int(off[e]), int(T[e])
            raw = r[s:s + t].astype(np.int64)
            turn = raw.copy()
            turn[1:] += raw[:-1]            # selfplay_worker.py:33-37: r[k] += original r[k-1]
            ep = {"game": int(games[e]), "vis": pol[s:s + t], "root": root[s:s + t].astype(np.float64),
                  "a": a[s:s + t].astype(np.int64), "r": turn, "r_raw": raw, "la": la[s + e:s + e + t + 1].astype(np.float64)}
            if store is None:
                ep["o"] = o[s + e * self.stack:s + e * self.stack + self.stack + t]
            else:
                ep["id"] = int(ids[e])
            out.append(ep)
        return out


class EpisodeRing:
    """Row bookkeeping of an EpisodeStore, on the host only.  One add places a contiguous block of rows: for episodes
    e = 0..E-1 with T_e moves, episode e's stack + T_e frames start at row base + off_e + e * stack and its T_e + 1
    legal rows at base + off_e + e (off_e = T_0 + ... + T_{e-1}), the layout hz_traj_pack writes, so the block takes
    sum(T) + E * stack rows of the frame arena and fewer of the legal arena.  Blocks follow one another around a ring of
    `capacity` rows; a block that does not fit before the end starts again at row 0, and the episodes the block
    overwrites are evicted, together with those left behind the wrap, so eviction always takes the oldest episodes
    first.  Ids are int64 and never reused; the live ids are one range [first, next_id)."""

    def __init__(self, capacity, stack):
        self.capacity, self.stack = int(capacity), int(stack)
        if not 1 <= self.capacity < 2 ** 31 or self.stack < 1:
            raise ValueError(f"capacity must be 1..2^31 - 1 rows and stack >= 1, got {capacity}, {stack}")
        self.head = 0                   # first row after the newest block
        self.first = self.next_id = 0   # live ids
        self._base = 0                  # id of entry 0 of the tables below
        self._frame = np.zeros(0, np.int64)
        self._legal = np.zeros(0, np.int64)
        self._len = np.zeros(0, np.int64)

    def __len__(self):
        return self.next_id - self.first

    def block_rows(self, T):
        T = np.asarray(T, np.int64)
        return int(T.sum()) + T.size * self.stack

    def add(self, T):
        """Places episodes of T[e] moves; returns (ids int64 [E], base row of the block).  Raises before changing
        anything when T is not a non-empty list of move counts or the block is larger than the ring."""
        T = np.asarray(T, np.int64).reshape(-1)
        if T.size == 0 or (T < 0).any():
            raise ValueError(f"an add takes one or more episodes with T >= 0 moves, got {T.tolist()}")
        size = int(T.sum()) + T.size * self.stack
        if size > self.capacity:
            raise ValueError(f"{T.size} episodes need {size} rows, more than the store's capacity of {self.capacity}")
        wrap = self.head + size > self.capacity
        base = 0 if wrap else self.head
        live = slice(self.first - self._base, self.next_id - self._base)
        lo, hi = self._legal[live], self._frame[live] + self.stack + self._len[live]    # each episode's rows [lo, hi)
        gone = ((lo < base + size) & (hi > base)) | (wrap & (lo >= self.head))
        # the evicted episodes are a prefix of the live ones (oldest first): count up to the first one kept
        self.first += int(np.argmin(gone)) if not gone.all() else int(gone.size)
        off = np.concatenate(([0], np.cumsum(T)[:-1])).astype(np.int64)
        e = np.arange(T.size, dtype=np.int64)
        keep = slice(self.first - self._base, None)
        self._frame = np.concatenate((self._frame[keep], base + off + e * self.stack))
        self._legal = np.concatenate((self._legal[keep], base + off + e))
        self._len = np.concatenate((self._len[keep], T))
        self._base = self.first
        ids = np.arange(self.next_id, self.next_id + T.size, dtype=np.int64)
        self.next_id += T.size
        self.head = base + size
        return ids, base

    def rows(self, ids):
        """(first frame row, first legal row, T) int64 arrays of live episodes; raises on an evicted or unknown id."""
        ids = np.asarray(ids, np.int64).reshape(-1)
        bad = (ids < self.first) | (ids >= self.next_id)
        if bad.any():
            raise ValueError(f"episode id {int(ids[bad][0])} is not in the store (evicted or never added; live ids "
                             f"{self.first}..{self.next_id - 1})")
        i = ids - self._base
        return self._frame[i], self._legal[i], self._len[i]

    def samples(self, ids, starts, positions):
        """hz_obs_pack_episodes' sample rows int32 [B, 4] for windows of `positions` positions from (id, start):
        {first window frame row, episode's last frame row, legal row of the start, positions with targets}.  Raises on
        an evicted or unknown id and on a start outside 0..T - 1."""
        ids = np.asarray(ids, np.int64).reshape(-1)
        starts = np.asarray(starts, np.int64).reshape(-1)
        if ids.shape != starts.shape:
            raise ValueError(f"ids and starts must have the same length, got {ids.size} and {starts.size}")
        frame, legal, T = self.rows(ids)
        bad = (starts < 0) | (starts >= T)
        if bad.any():
            k = int(np.flatnonzero(bad)[0])
            raise ValueError(f"start {int(starts[k])} of episode {int(ids[k])} is outside 0..T - 1 (T = {int(T[k])})")
        out = np.empty((ids.size, 4), np.int32)
        out[:, 0] = frame + starts
        out[:, 1] = frame + self.stack + T - 1
        out[:, 2] = legal + starts
        out[:, 3] = np.clip(T - starts, 0, int(positions))
        return out


class EpisodeStore:
    """Finished episodes kept in device memory for reanalyze: a byte frame arena uint8 [capacity, obs_dim] and a legal
    arena uint8 [capacity, num_actions] in the row layout of hz_traj_pack (`stack` copies of an episode's first frame,
    then one row per move; T + 1 legal rows), filled by TrajectoryRecorder.flush(store=...) / SelfPlayPool.flush(store=...)
    on the recording streams or by add() from flushed dicts, and read by ReanalyzePipeline.submit_episodes tickets that
    name (episode id, start).  Space is a ring of whole episodes (EpisodeRing): the oldest are evicted as new ones come.

    Ordering without host synchronisation: every add runs on the caller's current stream after the previous add (event)
    and after every pack launch that read an episode it evicts; a pack runs after the adds made before its ticket was
    submitted.  A ticket waiting in an open wave has no pack launch yet, so an add that evicts anything first launches
    the open waves that read this store (SearchPipeline.flush of the pipelines it has served).  Not thread-safe."""

    def __init__(self, capacity, obs_dim, num_actions, stack=4, device=None):
        import weakref
        self.ring = EpisodeRing(capacity, stack)
        self.capacity, self.obs_dim, self.num_actions, self.stack = self.ring.capacity, int(obs_dim), int(num_actions), self.ring.stack
        from .cytree import _device_index
        self.device = torch.device("cuda", _device_index(torch.cuda.current_device() if device is None else device))
        self.frames = torch.zeros(self.capacity, self.obs_dim, dtype=torch.uint8, device=self.device)
        self.legal = torch.zeros(self.capacity, self.num_actions, dtype=torch.uint8, device=self.device)
        self._last_add = None        # event recorded after the newest add
        self._readers = []           # (event after a pack launch, lowest id it read)
        self._pipes = weakref.WeakSet()

    def __len__(self):
        return len(self.ring)

    def samples(self, ids, starts, positions):
        return self.ring.samples(ids, starts, positions)

    def _check_recorder(self, rec):
        from .cytree import _device_index
        if ((rec.obs_dim, rec.actions, rec.stack, _device_index(rec.device))
                != (self.obs_dim, self.num_actions, self.stack, self.device.index)):
            raise ValueError(f"recorder (obs_dim {rec.obs_dim}, actions {rec.actions}, stack {rec.stack}, {rec.device}) "
                             f"does not fit the store (obs_dim {self.obs_dim}, actions {self.num_actions}, stack "
                             f"{self.stack}, {self.device})")

    def _watch(self, pipe):
        """A SearchPipeline took a ticket of this store: its open wave is launched before an add evicts anything."""
        self._pipes.add(pipe)

    def _read(self, event, low_id):
        """A pack launch read episodes from low_id on; `event` follows it on the reading stream."""
        self._readers.append((event, int(low_id)))

    def _begin_add(self, T):
        """Places the block (raising before any device work) and makes the current stream wait for what the add must
        follow.  Returns (ids, base row)."""
        first = self.ring.first
        ids, base = self.ring.add(T)
        st = torch.cuda.current_stream(self.device)
        if self.ring.first != first:
            for pipe in list(self._pipes):
                if pipe._open_reads(self):
                    pipe.flush()
        if self._last_add is not None:
            st.wait_event(self._last_add)
        kept = []
        for ev, low in self._readers:
            if low < self.ring.first:
                st.wait_event(ev)        # read an evicted episode; later adds follow this one
            else:
                kept.append((ev, low))
        self._readers = kept
        return ids, base

    def _end_add(self):
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        self._last_add = ev

    def add(self, episodes):
        """Episodes recorded elsewhere: dicts with 'o' uint8 [stack + T, obs_dim] and 'la' [T + 1, num_actions] 0/1
        (what TrajectoryRecorder.flush returns).  One H2D copy on the current stream; returns their ids (int64 [E])."""
        eps = list(episodes)
        if not eps:
            return np.zeros(0, np.int64)
        T = []
        for k, ep in enumerate(eps):
            o, la = np.asarray(ep["o"]), np.asarray(ep["la"])
            t = o.shape[0] - self.stack if o.ndim == 2 else -1
            if t < 0 or o.shape[1] != self.obs_dim or la.shape != (t + 1, self.num_actions):
                raise ValueError(f"episode {k}: 'o' must be [stack + T, {self.obs_dim}] and 'la' [T + 1, "
                                 f"{self.num_actions}], got {o.shape} and {la.shape}")
            T.append(t)
        size, lrows = self.ring.block_rows(T), sum(T) + len(T)
        if size > self.capacity:
            raise ValueError(f"{len(T)} episodes need {size} rows, more than the store's capacity of {self.capacity}")
        D, A = self.obs_dim, self.num_actions
        host = torch.empty(size * D + lrows * A, dtype=torch.uint8, pin_memory=True)
        h = host.numpy()
        h[:size * D].reshape(size, D)[:] = np.concatenate([np.asarray(ep["o"]) for ep in eps]) != 0
        h[size * D:].reshape(lrows, A)[:] = np.concatenate([np.asarray(ep["la"]) for ep in eps]) != 0
        ids, base = self._begin_add(T)
        staged = host.to(self.device, non_blocking=True)
        self.frames[base:base + size].copy_(staged[:size * D].view(size, D))
        self.legal[base:base + lrows].copy_(staged[size * D:].view(lrows, A))
        self._end_add()
        return ids
