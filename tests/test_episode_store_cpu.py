"""CPU: the parts of the episode store that need no device — the ctypes mirror of hz_obs_episode_ticket, the argument
checks of hz_obs_pack_episodes (nothing launched), the ring bookkeeping of EpisodeRing (placement, wrap, eviction order,
ids, oversize adds, the sample rows the pack reads) and ReanalyzePipeline.submit_episodes rejecting bad ids, starts and
stores before taking a ticket."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from helpers import ROOT
from test_reanalyze_pipeline_cpu import _Config, _layout, _pipeline


def test_episode_ticket_mirrors_the_header_layout(tmp_path):
    from hanabizero_b200 import _lib
    cls = _lib.EpisodeTicket
    lines = ['printf("%zu", sizeof(hz_obs_episode_ticket));']
    lines += [f'printf(" %zu", offsetof(hz_obs_episode_ticket, {f}));' for f, _ in cls._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hzb200.h"\nint main(void) {\n' + "\n".join(lines)
                   + "\nreturn 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert ctypes.sizeof(cls) == out[0] == 48
    assert [getattr(cls, f).offset for f, _ in cls._fields_] == out[1:] == [0, 8, 16, 24, 32, 40]
    assert 64 * ctypes.sizeof(cls) <= 4096       # the table travels in the kernel parameters


def _ticket(**over):
    from hanabizero_b200 import _lib
    f = dict(frames=0x1000, ld_frames=785, legal=0x2000, samples=0x3000, noise=None, mask=0x4000)
    f.update(over)
    return _lib.EpisodeTicket(**f)


def test_obs_pack_episodes_rejects_bad_arguments_before_touching_a_device():
    from hanabizero_b200 import _lib
    lib = _lib.load()
    before = lib.hz_launch_count()
    buf = ctypes.c_void_p(0x1000)

    def pack(tickets=None, count=1, slots=2, n=60, a=20, layout=None, positions=6, x=buf, legal=buf, table=True):
        tab = (_lib.EpisodeTicket * max(1, len(tickets or [0])))(*(tickets or [_ticket()])) if table else None
        lay = ctypes.byref(layout if layout is not None else _layout())
        return lib.hz_obs_pack_episodes(None, 0, tab, count, slots, n, a, lay, positions, x, legal, buf)

    cases = [
        (dict(table=False), b"NULL ticket table"),
        (dict(count=3), b"count"), (dict(count=0), b"count"), (dict(slots=65), b"slots"), (dict(slots=0), b"slots"),
        (dict(n=0), b"n = 0"), (dict(slots=64, n=1 << 19), b"slots * n"),
        (dict(n=62), b"not a multiple of positions"), (dict(positions=0), b"positions"),
        (dict(n=6, positions=12), b"positions"),
        (dict(a=33), b"num_actions"), (dict(a=0), b"num_actions"),
        (dict(layout=_layout(stack=0)), b"stack"), (dict(layout=_layout(stack=65)), b"stack"),
        (dict(layout=_layout(frame_stride=808)), b"frame_stride"),
        (dict(layout=_layout(frame_dim=801)), b"frame_dim"), (dict(layout=_layout(elem_bytes=1)), b"elem_bytes"),
        (dict(x=None), b"NULL staging"), (dict(legal=None), b"NULL staging"),
        (dict(tickets=[_ticket(frames=None)]), b"ticket 0 has a NULL input"),
        (dict(tickets=[_ticket(), _ticket(legal=None)], count=2), b"ticket 1 has a NULL input"),
        (dict(tickets=[_ticket(samples=None)]), b"ticket 0 has a NULL input"),
        (dict(tickets=[_ticket(mask=None)]), b"NULL mask"),
        (dict(tickets=[_ticket(ld_frames=784)]), b"ld_frames"),
    ]
    for kw, msg in cases:
        assert pack(**kw) == _lib.HZ_ERR_ARG, kw
        assert msg in lib.hz_last_error(), (kw, lib.hz_last_error())
    assert lib.hz_obs_pack_episodes(None, 0, (_lib.EpisodeTicket * 1)(_ticket()), 1, 1, 60, 20, None, 6, buf, buf,
                                    buf) == _lib.HZ_ERR_ARG
    assert b"NULL layout" in lib.hz_last_error()
    assert lib.hz_launch_count() == before


# ---- ring bookkeeping -----------------------------------------------------------------------------------------------

def _extent(ring, i):
    """Rows [lo, hi) episode i takes in the arenas (legal rows start first, frame rows end last)."""
    f, l, T = (int(v[0]) for v in ring.rows([i]))
    return l, f + ring.stack + T


def test_ring_places_blocks_contiguously_in_the_pack_layout():
    from hanabizero_b200.trajectory import EpisodeRing
    r = EpisodeRing(1000, 4)
    ids, base = r.add([10, 0, 7])
    assert ids.tolist() == [0, 1, 2] and base == 0 and r.head == 17 + 3 * 4
    frame, legal, T = r.rows(ids)
    # hz_traj_pack: frames of e at off_e + e * stack, legal rows at off_e + e
    assert frame.tolist() == [0, 14, 18] and legal.tolist() == [0, 11, 12] and T.tolist() == [10, 0, 7]
    ids, base = r.add([5])
    assert ids.tolist() == [3] and base == 29 and r.rows([3])[0].tolist() == [29] and r.rows([3])[1].tolist() == [29]
    assert len(r) == 4 and r.first == 0 and r.head == 38


def test_ring_wraps_and_evicts_the_oldest_episodes_first():
    from hanabizero_b200.trajectory import EpisodeRing
    rng = np.random.default_rng(0)
    cap, S = 500, 4
    r = EpisodeRing(cap, S)
    arena = np.full(cap, -1, np.int64)      # first id of the block that last wrote each row
    seen = set()
    for step in range(300):
        T = rng.integers(0, 40, rng.integers(1, 4)).tolist()
        head = r.head
        ids, base = r.add(T)
        size = sum(T) + len(T) * S
        assert base == (head if head + size <= cap else 0)
        assert not seen & set(ids.tolist())                       # never reused
        seen |= set(ids.tolist())
        assert ids.tolist() == list(range(r.next_id - len(T), r.next_id))
        # every live episode's rows are its own in the arena model
        arena[base:base + size] = ids[0]
        for i in ids.tolist():
            lo, hi = _extent(r, i)
            assert base <= lo < hi <= base + size
        for i in range(r.first, r.next_id):
            lo, hi = _extent(r, i)
            blk = arena[lo:hi]
            assert (blk == blk[0]).all() and blk[0] <= i and blk[0] > i - 4, (step, i)
        # eviction is oldest first: the live ids are a range ending at the newest
        assert r.first <= ids[0] and r.next_id == ids[-1] + 1
        for i in range(max(0, r.first - 5), r.first):
            with pytest.raises(ValueError, match="not in the store"):
                r.rows([i])
    assert r.first > 50             # the ring went round many times


def test_ring_evicts_whatever_a_wrapped_block_leaves_behind():
    from hanabizero_b200.trajectory import EpisodeRing
    r = EpisodeRing(100, 2)
    r.add([20])          # rows 0..22, id 0
    r.add([20])          # rows 22..44, id 1
    r.add([20])          # rows 44..66, id 2
    r.add([20])          # rows 66..88, id 3
    ids, base = r.add([20])       # 88 + 22 > 100: wraps to 0, overwrites id 0, and ids 1..3 are older than id 4
    assert base == 0 and ids.tolist() == [4]
    # the oldest episodes go first: id 0 overwritten; 1..3 survive until overwritten (they are not behind the wrap)
    assert r.first == 1
    ids, base = r.add([50])       # 22 + 52 <= 100: rows 22..74 evict ids 1..3 (3 ends at 88 but starts at 66 < 74)
    assert base == 22 and r.first == 4
    ids, base = r.add([20])       # 74 + 22 = 96 fits
    assert base == 74 and r.first == 4
    ids, base = r.add([10])       # 96 + 12 > 100: wraps; rows 0..12 overwrite id 4
    assert base == 0 and r.first == 5 and ids.tolist() == [7]
    r2 = EpisodeRing(100, 2)
    r2.add([30]), r2.add([30])      # 0..32, 32..64
    r2.add([30])                    # 64..96
    r2.add([40])                    # wraps, 0..42: evicts ids 0 and 1 (1 starts at 32 < 42)
    assert r2.first == 2 and r2.head == 42
    r2.add([50])                    # 42 + 52 = 94 fits: evicts id 2 (64..96)
    assert r2.first == 3
    r2.add([10])                    # 94 + 12 > 100: wraps, and nothing is left behind the wrap but the tail is empty
    assert r2.first == 3 + 1 and r2.head == 12      # id 3 (0..42) overwritten


def test_ring_rejects_an_oversize_add_without_changing_anything():
    from hanabizero_b200.trajectory import EpisodeRing
    r = EpisodeRing(100, 4)
    r.add([30, 20])
    state = (r.head, r.first, r.next_id)
    for T in ([97], [50, 43], [], [-1], [200]):
        with pytest.raises(ValueError):
            r.add(T)
        assert (r.head, r.first, r.next_id) == state
    ids, base = r.add([96])          # exactly the capacity
    assert base == 0 and r.first == 2 and ids.tolist() == [2]
    with pytest.raises(ValueError):
        EpisodeRing(0, 4)
    with pytest.raises(ValueError):
        EpisodeRing(10, 0)


def test_ring_sample_rows():
    from hanabizero_b200.trajectory import EpisodeRing
    S, P = 4, 6
    r = EpisodeRing(1000, S)
    r.add([12, 3])
    r.add([1])
    f, l, T = r.rows([0, 1, 2])
    got = r.samples([0, 0, 0, 1, 1, 2], [0, 6, 11, 0, 2, 0], P)
    assert got.dtype == np.int32 and got.shape == (6, 4)
    want = [
        [f[0] + 0, f[0] + S + 11, l[0] + 0, 6],
        [f[0] + 6, f[0] + S + 11, l[0] + 6, 6],
        [f[0] + 11, f[0] + S + 11, l[0] + 11, 1],     # start = T - 1: one position with a target
        [f[1] + 0, f[1] + S + 2, l[1] + 0, 3],        # shorter than K + 1 positions
        [f[1] + 2, f[1] + S + 2, l[1] + 2, 1],
        [f[2] + 0, f[2] + S + 0, l[2] + 0, 1],
    ]
    assert got.tolist() == [[int(v) for v in row] for row in want]
    for ids, starts in (([0], [12]), ([0], [-1]), ([1], [3]), ([2], [1]), ([3], [0]), ([-1], [0]), ([0, 1], [0])):
        with pytest.raises(ValueError):
            r.samples(ids, starts, P)


# ---- submit_episodes ------------------------------------------------------------------------------------------------

def _store(capacity=1000, obs_dim=785, num_actions=20, stack=4, device=torch.device("cuda", 0), T=(10,) * 6):
    """An EpisodeStore with only its bookkeeping (no device), holding episodes of T moves."""
    from hanabizero_b200.trajectory import EpisodeRing, EpisodeStore
    s = EpisodeStore.__new__(EpisodeStore)
    s.ring = EpisodeRing(capacity, stack)
    s.capacity, s.obs_dim, s.num_actions, s.stack, s.device = capacity, obs_dim, num_actions, stack, device
    s.ring.add(T)
    return s


def test_submit_episodes_rejects_bad_ids_starts_and_stores():
    from hanabizero_b200.reanalyze import ReanalyzePipeline
    batch, K, S, A = 4, 5, 4, 20
    rp = ReanalyzePipeline.__new__(ReanalyzePipeline)
    rp.config, rp.batch, rp.per, rp.stack, rp.a = _Config(), batch, K + 1, S, A
    rp.roots = batch * (K + 1)
    rp.pipe = _pipeline(n=rp.roots, stack=S)
    rp.device, rp._out = rp.pipe.device, {}
    store = _store(T=[10, 3, 7, 1])
    store.ring.add([800])                           # evicts nothing yet
    store.ring.add([200])                           # wraps: evicts ids 0..4
    assert store.ring.first == 5
    good = dict(store=_store(), ids=[0, 1, 2, 3], starts=[0, 9, 5, 3])
    bad = [
        dict(ids=[0, 1, 2, 6]), dict(ids=[0, 1, 2, -1]),                        # unknown
        dict(store=store, ids=[5, 5, 0, 5], starts=[0, 0, 0, 0]),              # evicted
        dict(starts=[0, 10, 5, 3]), dict(starts=[-1, 0, 0, 0]),                 # outside 0..T - 1
        dict(ids=[0, 1, 2]), dict(starts=[0, 1, 2, 3, 4]),                      # not [batch]
        dict(store=_store(obs_dim=660)), dict(store=_store(num_actions=11)), dict(store=_store(stack=2)),
        dict(store=_store(device=torch.device("cuda", 1))),
        dict(out=torch.zeros(batch, K + 1, A)), dict(out=torch.zeros(batch, K, A, dtype=torch.float64)),
        dict(noises=torch.zeros(batch * (K + 1), A + 1)),
    ]
    for kw in bad:
        args = dict(good)
        args.update(kw)
        with pytest.raises(ValueError):
            rp.submit_episodes(**args)
        assert rp.pipe._waves.open is None and rp.pipe.submitted == 0 and not rp._out, kw
