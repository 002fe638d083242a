"""GPU: the episode store.  Self-play flushed into a store against the same self-play flushed to the host (and added
with store.add), byte for byte; ReanalyzePipeline.submit_episodes targets against submit() of windows, legal rows and
masks cut from the flushed episodes on the host, bit for bit, over starts at both ends of episodes, short episodes,
full and partial waves, two stores in one wave and episode tickets between window tickets; targets on real positions
with 50 simulations; a ticket whose episode is evicted while its wave is still open; and self-play flushing into the
store while reanalyze tickets are in flight."""
import copy

import numpy as np
import pytest
import torch

from test_search_obs_gpu import _model as _net
from test_selfplay_record_gpu import GAMES, _model as _play_model

pytestmark = pytest.mark.gpu

S = 4


def _pool(game, mdp, engines=2, N=16, sims=6):
    from hanabizero_b200.mcts import SearchConfig
    from hanabizero_b200.selfplay import SelfPlayEngine, SelfPlayPool
    model = _play_model(game, mdp, S)
    cfg = SearchConfig(num_simulations=sims, amp_type="torch_amp")
    return SelfPlayPool([SelfPlayEngine(N, game, model, cfg, seeds=np.arange(N) + 100 * e, mdp=mdp, stack=S,
                                        record="ring", record_banks=4, noise_seed=3, game_offset=e * N)
                         for e in range(engines)])


def _play(pool, moves, flush_every, store=None):
    """Steps the pool deterministically, flushing every `flush_every` moves; returns every flushed dict in order."""
    eps = []
    pool.reset()
    for m in range(moves):
        pool.step(deterministic=True)
        if m % flush_every == flush_every - 1:
            for e in pool.flush(store=store):
                eps += e
    pool.check()
    return eps


_EPISODES = {}


def _episodes(game="Hanabi-Full", mdp="global"):
    """Host-flushed episodes of a small self-play run (cached per game)."""
    if (game, mdp) not in _EPISODES:
        _EPISODES[game, mdp] = _play(_pool(game, mdp), 60, 3)     # banks - 1 moves at most
    return _EPISODES[game, mdp]


def _store(capacity, game="Hanabi-Full", mdp="global"):
    from hanabizero_b200.trajectory import EpisodeStore
    return EpisodeStore(capacity, GAMES[game]["dims"][mdp], GAMES[game]["A"], S)


def _rows(store, i):
    """(frames, legal rows) of episode i, copied from the store's arenas."""
    f, l, T = (int(v[0]) for v in store.ring.rows([i]))
    return store.frames[f:f + S + T].cpu().numpy(), store.legal[l:l + T + 1].cpu().numpy()


@pytest.mark.parametrize("game,mdp", [("Hanabi-Full", "global"), ("Hanabi-Small", "local")])
def test_flush_into_the_store_equals_the_host_flush(game, mdp):
    """Two identical pools, one flushed to the host and one into a store: the store's rows equal 'o' and 'la' bit for
    bit, every other key is unchanged, and store.add of the host dicts puts the same rows into another store."""
    host = _episodes(game, mdp)
    store = _store(1 << 16, game, mdp)
    dev = _play(_pool(game, mdp), 60, 3, store=store)
    torch.cuda.synchronize()
    assert len(host) == len(dev) and len(host) >= 16 and len(store) == len(dev)
    added = _store(1 << 16, game, mdp)
    ids = added.add(host[:len(host) // 2])
    ids = np.concatenate((ids, added.add(host[len(host) // 2:])))
    torch.cuda.synchronize()
    assert ids.tolist() == list(range(len(host)))
    for k, (h, d) in enumerate(zip(host, dev)):
        assert set(d) == set(h) - {"o"} | {"id"} and d["id"] == k
        for key in h:
            if key != "o":
                assert np.array_equal(h[key], d[key]) and np.asarray(h[key]).dtype == np.asarray(d[key]).dtype, (k, key)
        for s in (store, added):
            o, la = _rows(s, k)
            assert np.array_equal(o, h["o"]) and np.array_equal(la, h["la"]), k


# ---- targets ----------------------------------------------------------------------------------------------------------

def _cut(ep, start, K):
    """The host path: the window of frames start .. start + K + S - 1 (clamped to the episode's last frame), the legal
    rows of positions start .. start + K (zero past the end) and their mask."""
    o, la, T = ep["o"], ep["la"], len(ep["a"])
    win = o[np.minimum(start + np.arange(K + S), S + T - 1)]
    pos = start + np.arange(K + 1)
    keep = pos < T
    legal = np.where(keep[:, None], la[np.minimum(pos, T)], 0).astype(np.float32)
    return win, legal, keep.astype(np.uint8)


def _host_ticket(eps, picks, K):
    cut = [_cut(eps[i], s, K) for i, s in picks]
    return [torch.from_numpy(np.stack(x)).cuda() for x in zip(*cut)]


def _picks(eps, batch, K, seed, ids=None):
    """(episode index, start) per sample: both ends of episodes, episodes shorter than K + 1 positions, random starts."""
    rng = np.random.default_rng(seed)
    ids = np.arange(len(eps)) if ids is None else np.asarray(ids)
    T = np.array([len(eps[i]["a"]) for i in ids])
    short = ids[T < K + 1]
    out = []
    for b in range(batch):
        i = int(ids[rng.integers(len(ids))]) if b % 4 or not len(short) else int(short[rng.integers(len(short))])
        t = len(eps[i]["a"])
        out.append((i, [0, t - 1, int(rng.integers(t)), max(0, t - K)][b % 4]))
    return out


def _pipe(batch, K, wave, depth=2, sims=12):
    from hanabizero_b200.mcts import SearchConfig
    from hanabizero_b200.reanalyze import ReanalyzePipeline
    cfg = SearchConfig(num_simulations=sims, amp_type="torch_amp")
    cfg.action_space_size = 20
    rp = ReanalyzePipeline(cfg, _net(True, 785, S, 20, seed=4), batch, K, S, depth=depth, wave=wave)
    assert rp.pipe.executor == "rows"          # every ticket's trees alone, whatever else its wave holds
    return rp


def _same(a, b):
    return torch.equal(a.reshape(-1).view(torch.int64), b.reshape(-1).view(torch.int64))


def test_episode_targets_equal_the_host_path():
    """Tickets from two stores (holding the same episodes at different rows), mixed in waves of 3 with window tickets
    in between (which launch the open wave: partial waves), against submit() of host-cut windows in a pipeline of its
    own: equal bit for bit, masked rows zero, kept rows summing to 1."""
    batch, K, G = 24, 5, 3
    eps = _episodes() + [dict(e, o=e["o"][:S + t], la=e["la"][:t + 1], a=e["a"][:t]) for t in (1, 2, 4)
                         for e in _episodes()[:2]]      # real frames cut short: episodes of fewer than K + 1 moves
    A = [_store(1 << 15), _store(1 << 15)]
    ids_a = A[0].add(eps)
    A[1].add(eps[:3])                              # other rows for the same episodes
    ids_b = A[1].add(eps)
    assert ids_a.tolist() == list(range(len(eps))) and ids_b[0] == 3
    rp, ref = _pipe(batch, K, G, depth=8), _pipe(batch, K, G, depth=8)      # no slot reused before the results
    plan = ["a", "b", "a", "a", "win", "b", "a", "win", "win", "b", "b", "a", "b"]
    got, want = [], []
    for k, kind in enumerate(plan):
        picks = _picks(eps, batch, K, seed=k)
        assert min(len(eps[i]["a"]) for i, _ in picks) < K + 1
        win, legal, mask = _host_ticket(eps, picks, K)
        if kind == "win":
            got.append(rp.submit(win, legal, mask, noise_seed=2, noise_step=k))
        else:
            st, ids = (A[0], ids_a) if kind == "a" else (A[1], ids_b)
            got.append(rp.submit_episodes(st, [int(ids[i]) for i, _ in picks], [s for _, s in picks], noise_seed=2,
                                          noise_step=k))
        want.append((ref.submit(win, legal, mask, noise_seed=2, noise_step=k), mask))
    rp.drain()
    for k, (t, (u, mask)) in enumerate(zip(got, want)):
        g, w = rp.result(t).reshape(-1, 20), ref.result(u).reshape(-1, 20)
        assert _same(g, w), (k, plan[k])
        m = mask.reshape(-1).bool()
        assert not g[~m].any() and float((g[m].sum(1) - 1).abs().max()) < 1e-12, k
    assert sum(int((m == 0).sum()) for _, m in want) > 0


def test_episode_targets_on_real_positions():
    """50 simulations over self-play positions read from a store flushed by the pool: every kept row sums to 1 within
    1e-12 and rows past the end of an episode are zero."""
    store = _store(1 << 16)
    eps = _play(_pool("Hanabi-Full", "global"), 60, 3, store=store)
    batch, K = 128, 5
    rp = _pipe(batch, K, wave=1, sims=50)
    rng = np.random.default_rng(1)
    ids = rng.integers(0, len(eps), batch)
    T = np.array([len(eps[i]["a"]) for i in ids])
    starts = np.where(np.arange(batch) % 3 == 0, T - 1, rng.integers(0, T))
    got = rp.result(rp.submit_episodes(store, [eps[i]["id"] for i in ids], starts, noise_seed=1)).reshape(-1, 20)
    keep = torch.from_numpy(((starts[:, None] + np.arange(K + 1)) < T[:, None]).reshape(-1)).cuda()
    assert not got[~keep].any() and bool((~keep).any())
    assert float((got[keep].sum(1) - 1).abs().max()) < 1e-12


def test_a_ticket_survives_the_eviction_of_its_episode():
    """A ticket waits in an open wave while adds evict its episodes and overwrite their rows: the add launches the wave
    first and waits for its pack, so the targets are those of the original data.  Then the evicted id raises."""
    eps = _episodes()
    batch, K, G = 16, 5, 3
    rows = sum(len(e["o"]) for e in eps)
    store = _store(rows + 8)
    ids = store.add(eps)
    rp, ref = _pipe(batch, K, G), _pipe(batch, K, G)
    picks = _picks(eps, batch, K, seed=9)
    t = rp.submit_episodes(store, [int(ids[i]) for i, _ in picks], [s for _, s in picks], noise_seed=4)
    assert rp.pipe._waves.open is not None                       # the wave is still open: no pack yet
    other = [dict(e, o=np.ones_like(e["o"]), la=np.ones_like(e["la"])) for e in eps[::-1][:len(eps) // 2]]
    new = store.add(other)                                       # wraps to row 0 and evicts the oldest episodes
    assert rp.pipe._waves.open is None and store.ring.first > 0
    win, legal, mask = _host_ticket(eps, picks, K)
    want = ref.result(ref.submit(win, legal, mask, noise_seed=4))
    assert _same(rp.result(t), want)
    torch.cuda.synchronize()
    f, _, _ = store.ring.rows([int(new[0])])
    assert int(f[0]) == 0 and bool(store.frames[:len(other[0]["o"])].eq(1).all())   # the rows were overwritten
    gone = next(int(ids[i]) for i, _ in picks if ids[i] < store.ring.first)
    with pytest.raises(ValueError, match="not in the store"):
        rp.submit_episodes(store, [gone] * batch, [0] * batch)


def test_tickets_in_flight_while_self_play_flushes_into_the_store():
    """Self-play keeps stepping and flushing into the store on its engines' streams (evicting the oldest episodes) while
    reanalyze tickets on its episodes are in flight: every result equals the same ticket run against a quiet copy of
    the store."""
    from hanabizero_b200.trajectory import EpisodeStore
    pool = _pool("Hanabi-Full", "global", engines=2, N=16)
    per_move = sum(len(e["o"]) for e in _episodes()) / 60        # rows the pool adds per move, about
    store = _store(int(per_move * 40))                           # 30 moves fill three quarters of it
    eps = []
    pool.reset()
    for m in range(30):
        pool.step(deterministic=True)
        if m % 3 == 2:
            for e in pool.flush(store=store):
                eps += e
    torch.cuda.synchronize()
    quiet = EpisodeStore(store.capacity, store.obs_dim, store.num_actions, S)
    quiet.frames.copy_(store.frames)
    quiet.legal.copy_(store.legal)
    quiet.ring = copy.deepcopy(store.ring)
    torch.cuda.synchronize()
    live = (store.ring.first, store.ring.next_id)
    batch, K, G, lag = 16, 5, 2, 3
    rp = _pipe(batch, K, G, depth=4)
    byid = {e["id"]: e for e in eps}
    tickets, got = [], []
    for k in range(12):
        lo = max(live[0], store.ring.first)
        if lo >= live[1]:
            break
        ids = list(range(lo, live[1]))
        picks = _picks([byid[i] for i in ids], batch, K, seed=20 + k)
        args = ([ids[i] for i, _ in picks], [s for _, s in picks])
        tickets.append((rp.submit_episodes(store, *args, noise_seed=6, noise_step=k), args, k))
        pool.step(deterministic=True)
        for _ in pool.flush(store=store):
            pass
        pool.step(deterministic=True)
        if len(tickets) > lag:          # consumed before its slot is taken again
            t, a, j = tickets.pop(0)
            got.append((rp.result(t).clone(), a, j))
    got += [(rp.result(t).clone(), a, j) for t, a, j in tickets]
    assert store.ring.first > live[0] and len(got) >= 4          # episodes the tickets read were evicted
    pool.synchronize()
    calm = _pipe(batch, K, G, depth=3)
    for g, args, k in got:
        assert _same(g, calm.result(calm.submit_episodes(quiet, *args, noise_seed=6, noise_step=k))), k
