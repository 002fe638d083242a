"""GPU: search waves (SearchPipeline(wave=G), hz_wave_pack / hz_wave_unpack).  G tickets of n roots searched as one
batch of G * n trees must give every ticket exactly its own rows: on the row-block executor, bit for bit what a
stand-alone Roots(n) + run_multi of that ticket alone gives (k_row_chain computes every row on its own, and the tree,
prepare and statistics kernels work per tree); on the library chain, bit for bit one run_multi over the concatenated
batch.  Padding rows of partial waves must not leak into any ticket."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

S = 12


def _cfg():
    from hanabizero_b200.mcts import SearchConfig
    return SearchConfig(num_simulations=S, amp_type="torch_amp")


def _model(full):
    from hanabizero_b200.model import MuZeroNet, MuZeroNetFull
    torch.manual_seed(0)
    if full:
        return MuZeroNetFull(785 * 4, 20).randomize_heads(std=0.05).to("cuda").eval(), 20
    return MuZeroNet(193 * 4, 11).randomize_heads(std=0.05).to("cuda").eval(), 11


def _ticket(n, a, seed, noisy=True, half=False):
    """Device inputs of one ticket, all different per seed; half=True gives the hidden state in the pool's fp16."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    rng = np.random.default_rng(seed)
    legal = (torch.rand(n, a, device="cuda", generator=g) < 0.6).int()
    legal[:, seed % a] = 1
    hidden = torch.randn(n, 512, device="cuda", generator=g).clamp_min(0) * 0.7
    return dict(noise=torch.from_numpy(rng.dirichlet([0.3] * a, n).astype(np.float32)).cuda() if noisy else None,
                reward=torch.randn(n, device="cuda", generator=g) * 0.1,
                logits=torch.randn(n, a, device="cuda", generator=g),
                legal=legal, hidden=hidden.half() if half else hidden,
                visits=torch.full((n, a), -1, dtype=torch.int32, device="cuda"),
                values=torch.full((n,), float("nan"), device="cuda"))


def _submit(pipe, t, fraction=0.25):
    return pipe.submit(fraction, t["noise"], t["reward"], t["logits"], t["legal"], t["hidden"], t["visits"], t["values"])


def _alone(mcts, model, t, n, a, fraction=0.25, **kw):
    """Stand-alone search of one ticket: Roots(n).prepare + run_multi."""
    from hanabizero_b200 import cytree
    roots = cytree.Roots(n, a, S)
    if t["noise"] is None:
        roots.prepare_no_noise(t["reward"], t["logits"], t["legal"])
    else:
        roots.prepare(fraction, t["noise"], t["reward"], t["logits"], t["legal"])
    mcts.run_multi(roots, model, t["hidden"], **kw)
    return roots.get_stats_tensors()


def _assert_equal(t, ref, what=""):
    v, val = ref
    assert torch.equal(t["visits"].cpu(), v.cpu()), what
    assert torch.equal(t["values"].cpu().view(torch.int32), val.cpu().view(torch.int32)), what


@pytest.mark.parametrize("full", [True, False], ids=["full", "small"])
@pytest.mark.parametrize("G", [2, 8])
@pytest.mark.parametrize("n", [128, 300, 512])
def test_wave_tickets_equal_their_stand_alone_row_searches(full, G, n):
    """Three full waves per slot (eager search, capture, replays); every third wave without noise; hidden states
    in fp32 (converted on the caller's stream) and in the pool's fp16 (read in place) alike."""
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    model, a = _model(full)
    depth = 2
    pipe = SearchPipeline(MCTS(_cfg()), model, n, a, depth=depth, executor="rows", wave=G)
    assert pipe.executor == "rows" and pipe.slots[0]["roots"].root_num == G * n
    tickets, ids = [], []
    for w in range(3 * depth):
        for p in range(G):
            t = _ticket(n, a, seed=1000 * w + p, noisy=w % 3 != 2, half=p % 2 == 1)
            ids.append(_submit(pipe, t))
            tickets.append(t)
    pipe.drain()
    torch.cuda.synchronize()
    assert ids == [(w % depth) * G + p for w in range(3 * depth) for p in range(G)]
    assert all(ws.chain._use_rows for ws in pipe.mcts._ws.values())
    ref = MCTS(_cfg())
    for k, t in enumerate(tickets):
        _assert_equal(t, _alone(ref, model, t, n, a, executor="rows"), k)
        assert int(t["visits"].sum()) == n * (S - 1)


def test_partial_waves_and_waits_on_unlaunched_waves():
    """flush() with 1 and G-1 tickets, wait() and stats() on a ticket of a wave that has not launched, and a change
    of noise-ness or fraction closing the open wave: every ticket still equals its stand-alone search (padding roots
    have no legal action and leak nothing)."""
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    model, a = _model(True)
    n, G = 300, 4
    pipe = SearchPipeline(MCTS(_cfg()), model, n, a, depth=2, executor="rows", wave=G)
    ref = MCTS(_cfg())
    done = []

    t = _ticket(n, a, 1)
    tid = _submit(pipe, t)
    pipe.flush()                                            # a wave of 1
    pipe.wait(tid)
    done.append((t, 0.25))
    group = [_ticket(n, a, 10 + p) for p in range(G - 1)]
    ids = [_submit(pipe, x) for x in group]
    pipe.flush()                                            # a wave of G - 1
    done += [(x, 0.25) for x in group]
    for rnd in range(3):                                    # waves closed by wait() / stats() on an open wave
        t = _ticket(n, a, 100 + rnd, noisy=rnd != 1)
        tid = _submit(pipe, t)
        if rnd == 2:
            v, val = pipe.stats(tid)
            torch.cuda.current_stream().synchronize()
            assert v.shape == (n, a) and int(v.sum()) == n * (S - 1)
        pipe.wait(tid)
        _assert_equal(t, _alone(ref, model, t, n, a, executor="rows"), ("wait", rnd))
    mixed = [(_ticket(n, a, 200), 0.25), (_ticket(n, a, 201, noisy=False), 0.25), (_ticket(n, a, 202), 0.25),
             (_ticket(n, a, 203), 0.5)]                      # each closes the wave before it
    for x, f in mixed:
        _submit(pipe, x, fraction=f)
    pipe.drain()
    torch.cuda.synchronize()
    assert ids == [pipe.wave * 1 + p for p in range(G - 1)]
    for k, (x, f) in enumerate(done + mixed):
        _assert_equal(x, _alone(ref, model, x, n, a, fraction=f, executor="rows"), k)


def test_rejected_submit_leaves_the_open_wave_intact_and_device_cuda_writes_in_place():
    """A submit with a wrong-shaped input or output raises before the ticket takes a position: the tickets around it
    keep consecutive ids and their own rows.  A pipeline built with device='cuda' (no index) reads and writes device
    tensors in place."""
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    model, a = _model(True)
    n, G = 128, 4
    pipe = SearchPipeline(MCTS(_cfg()), model, n, a, depth=2, executor="rows", wave=G, device="cuda")
    assert pipe.device.index is not None
    good = [_ticket(n, a, 300 + p) for p in range(G)]
    ids = [_submit(pipe, good[0])]
    bad = dict(_ticket(n, a, 399), hidden=torch.zeros(n + 1, 512, device="cuda"))
    with pytest.raises(ValueError):
        _submit(pipe, bad)
    with pytest.raises(ValueError):
        _submit(pipe, dict(_ticket(n, a, 398), visits=torch.empty(n, a + 1, dtype=torch.int32, device="cuda")))
    ids.append(_submit(pipe, good[1]))
    slot = pipe.slots[0]
    assert len(slot["table"]) == 2 and slot["post"] == [] and pipe._waves.open["count"] == 2
    ids += [_submit(pipe, t) for t in good[2:]]
    pipe.drain()
    torch.cuda.synchronize()
    assert ids == list(range(G))
    ref = MCTS(_cfg())
    for k, t in enumerate(good):
        _assert_equal(t, _alone(ref, model, t, n, a, executor="rows"), k)


def test_pinned_host_device_and_pageable_inputs_in_one_wave():
    """Pinned-host and device inputs and outputs in one wave (read and written by the kernels in place), pageable host
    inputs and outputs and a float legal mask (the torch slow path): all equal their stand-alone searches."""
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    model, a = _model(True)
    n, G = 256, 4
    pipe = SearchPipeline(MCTS(_cfg()), model, n, a, depth=2, executor="rows", wave=G)
    ref = MCTS(_cfg())
    pinned = lambda x: None if x is None else x.cpu().pin_memory()
    pageable = lambda x: None if x is None else x.cpu()
    jobs = []
    for w in range(4):
        for p in range(G):
            t = _ticket(n, a, 50 * w + p, half=p == 1)
            kind = (w + p) % 4
            if kind == 1:
                t = {k: pinned(v) for k, v in t.items()}
            elif kind == 2:
                t = {k: pageable(v) for k, v in t.items()}
            elif kind == 3:
                t.update(noise=pinned(t["noise"]), legal=t["legal"].float(), visits=pinned(t["visits"]),
                         values=pageable(t["values"]))
            _submit(pipe, t)
            jobs.append(t)
    pipe.drain()
    torch.cuda.synchronize()
    dev = lambda x: None if x is None else x.cuda()
    for k, t in enumerate(jobs):
        ref_in = {key: dev(v) for key, v in t.items()}
        _assert_equal(t, _alone(ref, model, ref_in, n, a, executor="rows"), k)


def test_library_chain_wave_equals_one_search_over_the_concatenated_batch():
    from hanabizero_b200 import cytree
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    model, a = _model(True)
    n, G = 256, 4
    pipe = SearchPipeline(MCTS(_cfg()), model, n, a, depth=2, executor="library", wave=G)
    waves = [[_ticket(n, a, 10 * w + p) for p in range(G)] for w in range(4)]
    for wave in waves:
        for t in wave:
            _submit(pipe, t)
    pipe.drain()
    torch.cuda.synchronize()
    ref = MCTS(_cfg())
    for wave in waves:
        cat = lambda k: torch.cat([t[k] for t in wave])
        roots = cytree.Roots(G * n, a, S)
        roots.prepare(0.25, cat("noise"), cat("reward"), cat("logits"), cat("legal"))
        ref.run_multi(roots, model, cat("hidden"), gemm_sm_target=pipe.gemm_sm_target, stage_limit=pipe.stage_limit,
                      executor="library")
        v, val = roots.get_stats_tensors()
        assert torch.equal(cat("visits"), v) and torch.equal(cat("values").view(torch.int32), val.view(torch.int32))


def test_gathered_ticket_rows_with_world_size_one():
    from hanabizero_b200.dist import AsyncStatsGather
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    model, a = _model(False)
    n, G, depth = 128, 4, 2
    gather = AsyncStatsGather(G * n, a, torch.device("cuda"), depth=depth)
    with pytest.raises(ValueError):
        SearchPipeline(MCTS(_cfg()), model, n, a, depth=depth, gather=AsyncStatsGather(n, a, torch.device("cuda"),
                                                                                       depth=depth), wave=G)
    pipe = SearchPipeline(MCTS(_cfg()), model, n, a, depth=depth, executor="rows", gather=gather, wave=G)
    for w in range(2 * depth + 1):
        ids = [_submit(pipe, _ticket(n, a, 7 * w + p)) for p in range(G - (w == 2 * depth))]
        for tid in ids:
            v, val = pipe.stats(tid)
            gv, gval = pipe.gathered(tid)
            assert gv.shape == (n, a) and torch.equal(gv, v) and torch.equal(gval.view(torch.int32), val.view(torch.int32))
    pipe.drain()


def test_wave_abi_rejects_bad_pointers_without_launching():
    """A pageable pointer, a pointer of another device and a misaligned hidden state are argument errors, found
    before anything is launched."""
    from hanabizero_b200 import _lib
    lib = _lib.load()
    n, a, F = 64, 20, 256
    dev = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, device="cuda")
    stage = dict(noise=dev(n, a), reward=dev(n), logits=dev(n, a), legal=dev(n, a, dtype=torch.int32),
                 hidden=dev(n, F), stats=dev(n * (a + 1), dtype=torch.int32))
    src = dict(noise=dev(n, a), reward=dev(n), logits=dev(n, a), legal=dev(n, a, dtype=torch.int32), hidden=dev(n + 1, F),
               visits=dev(n, a, dtype=torch.int32), values=dev(n))
    st = torch.cuda.current_stream().cuda_stream

    def ticket(**over):
        t = _lib.WaveTicket()
        for k, f in (("noise", "noise"), ("reward", "reward"), ("logits", "logits"), ("legal", "legal"),
                     ("hidden", "hidden"), ("visits", "out_visits"), ("values", "out_values")):
            setattr(t, f, over.get(k, src[k].data_ptr()))
        return (_lib.WaveTicket * 1)(t)

    def pack(table):
        return lib.hz_wave_pack(st, 0, table, 1, 1, n, a, F * 4, stage["noise"].data_ptr(), stage["reward"].data_ptr(),
                                stage["logits"].data_ptr(), stage["legal"].data_ptr(), stage["hidden"].data_ptr())

    def unpack(table):
        return lib.hz_wave_unpack(st, 0, table, 1, 1, n, a, stage["stats"].data_ptr())

    assert pack(ticket()) == _lib.HZ_OK and unpack(ticket()) == _lib.HZ_OK
    torch.cuda.synchronize()
    before = lib.hz_launch_count()
    pageable = torch.zeros(n, a)
    assert pack(ticket(logits=pageable.data_ptr())) == _lib.HZ_ERR_ARG
    assert b"page-locked" in lib.hz_last_error()
    assert unpack(ticket(visits=torch.zeros(n, a, dtype=torch.int32).data_ptr())) == _lib.HZ_ERR_ARG
    assert pack(ticket(hidden=src["hidden"].data_ptr() + 4)) == _lib.HZ_ERR_ARG
    assert b"aligned" in lib.hz_last_error()
    if torch.cuda.device_count() > 1:
        other = torch.zeros(n, a, device="cuda:1")
        assert pack(ticket(noise=other.data_ptr())) == _lib.HZ_ERR_ARG
        assert b"device 1" in lib.hz_last_error()
        assert unpack(ticket(values=other.data_ptr())) == _lib.HZ_ERR_ARG
    assert lib.hz_launch_count() == before
    torch.cuda.synchronize()
