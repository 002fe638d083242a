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

    def flush(self):
        """Hand the finished episodes to the host.  Returns a list of dicts, one per episode, in the layout of
        GameHistory.save_file (game.py:136-140) after SelfPlay `put` (selfplay_worker.py:29-39):
          'game' int, 'vis' float64 [T, A], 'root' float64 [T], 'a' int64 [T], 'o' uint8 [stack + T, D],
          'r' int64 [T] turn rewards, 'r_raw' int64 [T] env rewards, 'la' float64 [T + 1, A].
        One small D2H (flags + lengths), one pack kernel, one D2H of the packed episodes."""
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
        o = torch.empty(total + E * self.stack, self.obs_dim, dtype=torch.uint8, device=dev)
        la = torch.empty(total + E, self.actions, dtype=torch.uint8, device=dev)
        a = torch.empty(total, dtype=torch.int32, device=dev)
        r = torch.empty(total, dtype=torch.int32, device=dev)
        vis = torch.empty(total, self.actions, dtype=torch.int32, device=dev)
        root = torch.empty(total, dtype=torch.float32, device=dev)
        check(self._lib.hz_traj_pack(self._stream(), self._ref, E, ptr(idx[0]), ptr(idx[1]), ptr(d_off), ptr(o),
                                     ptr(la), ptr(a), ptr(r), ptr(vis), ptr(root)))
        pol = torch.empty(total, self.actions, dtype=torch.float64, device=dev)
        if total:
            check(self._lib.hz_visit_policy(self._stream(), ptr(vis), None, total, self.actions, ptr(pol), None))
        o, la, a, r, pol, root = (x.cpu().numpy() for x in (o, la, a, r, pol, root))
        out = []
        for e in range(E):
            s, t = int(off[e]), int(T[e])
            raw = r[s:s + t].astype(np.int64)
            turn = raw.copy()
            turn[1:] += raw[:-1]            # selfplay_worker.py:33-37: r[k] += original r[k-1]
            out.append({"game": int(games[e]), "vis": pol[s:s + t], "root": root[s:s + t].astype(np.float64),
                        "a": a[s:s + t].astype(np.int64), "o": o[s + e * self.stack:s + e * self.stack + self.stack + t],
                        "r": turn, "r_raw": raw, "la": la[s + e:s + e + t + 1].astype(np.float64)})
        return out
