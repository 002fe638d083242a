"""GPU: hz_trees_search_step (the production launch: raw support logits in, one launch per simulation)
against the generic calls it fuses — hz_support_decode + hz_trees_backprop_traverse + a torch gather —
on synthetic network outputs.  Bit-exact trees and hand-off batches, including the register-q variants
(capacity <= 64 and > 64) and the deep-path fallback (path longer than a warp)."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import CONST, bits_equal, tree_inputs

pytestmark = pytest.mark.gpu


def _run(N, A, S, width, dtype, deep=False, seed=0):
    from hanabizero_b200 import _lib, cytree
    lib = _lib.load()
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev).manual_seed(seed)
    F, OH = 512, 32 if A > 16 else 16
    P3 = (width + 7) // 8 * 8
    d = tree_inputs(N, A, S, seed)
    if deep:   # one forced line of play: path length grows by one every simulation
        d["logits"][:] = -30.0
        d["logits"][:, 0] = 30.0
        d["mask"][:] = 1
    support = (torch.arange(width, device=dev, dtype=torch.float32) - (width - 1) // 2)
    outs = []
    for x in range(S):
        o = torch.randn(3, N, P3, device=dev, generator=gen)
        if deep:
            o[2, :, :] = -30.0
            o[2, :, 0] = 30.0
            o[0, :, :] = -20.0
            o[0, :, (width - 1) // 2 + 3 + (x % 3)] = 20.0      # value ~ +3..5: the line stays attractive
            o[1, :, :] = -20.0
            o[1, :, (width - 1) // 2] = 20.0                    # reward 0
        outs.append(o.to(dtype))
    states = [torch.rand(N, F, device=dev, generator=gen).to(dtype) for _ in range(S)]
    root_hidden = torch.rand(N, F, device=dev, generator=gen).to(dtype)
    eb = outs[0].element_size()
    st = torch.cuda.current_stream().cuda_stream
    results = []
    for fused in (True, False):
        roots = cytree.Roots(N, A, S)
        roots.prepare(CONST["frac"], d["noise"], d["reward"], d["logits"], d["mask"])
        mm = cytree.MinMaxStatsList(N)
        mm.set_delta(CONST["delta"])
        mmt = mm.tensor(dev)
        pool = torch.zeros(S + 1, N, F, device=dev, dtype=dtype)
        pool[0] = root_hidden
        batch = torch.zeros(N, F + OH, device=dev, dtype=dtype)
        ix = torch.zeros(N, dtype=torch.int32, device=dev)
        la = torch.zeros(N, dtype=torch.int32, device=dev)
        trace = []
        if fused:
            io = _lib.SearchIO()
            cur = torch.zeros(3, N, P3, device=dev, dtype=dtype)
            state = torch.zeros(N, F, device=dev, dtype=dtype)
            io.value_logits, io.ld_value = cur[0].data_ptr(), P3
            io.reward_logits, io.ld_reward = cur[1].data_ptr(), P3
            io.policy_logits, io.ld_policy = cur[2].data_ptr(), P3
            io.next_state, io.ld_state = state.data_ptr(), F
            io.support, io.support_width, io.support_delta = support.data_ptr(), width, 1.0
            io.elem_bytes, io.sanitize_nan = eb, 1
            io.pool, io.state_cols = pool.data_ptr(), F
            io.out_batch, io.ld_batch, io.onehot_cols = batch.data_ptr(), F + OH, OH
            io.out_ix, io.out_action = ix.data_ptr(), la.data_ptr()
            io.minmax, io.value_delta_max = mmt.data_ptr(), CONST["delta"]
            io.discount, io.pb_c_base, io.pb_c_init = CONST["discount"], CONST["pb_c_base"], CONST["pb_c_init"]
            ref = ctypes.byref(io)
            _lib.check(lib.hz_trees_search_step(roots.handle, st, 0, 1, ref))
            trace.append((ix.clone(), la.clone(), batch.clone()))
            for x in range(1, S):
                cur.copy_(outs[x])
                state.copy_(states[x])
                _lib.check(lib.hz_trees_search_step(roots.handle, st, x, 1 if x < S - 1 else 0, ref))
                if x < S - 1:
                    trace.append((ix.clone(), la.clone(), batch.clone()))
        else:
            hidden = torch.zeros(N, F, device=dev, dtype=dtype)
            dec = torch.zeros(2 * N, device=dev)

            def record():
                b = torch.zeros(N, F + OH, device=dev, dtype=dtype)
                b[:, :F] = hidden
                b[torch.arange(N, device=dev), F + la.long()] = 1.0
                trace.append((ix.clone(), la.clone(), b))

            _lib.check(lib.hz_trees_traverse(roots.handle, st, CONST["pb_c_base"], CONST["pb_c_init"], CONST["discount"],
                                             mmt.data_ptr(), CONST["delta"], ix.data_ptr(), None, la.data_ptr(), None,
                                             pool.data_ptr(), hidden.data_ptr(), F * eb))
            record()
            for x in range(1, S):
                vr = outs[x][:2].reshape(2 * N, P3)
                _lib.check(lib.hz_support_decode(st, vr.data_ptr(), eb, support.data_ptr(), dec.data_ptr(), 2 * N, width, P3, 1.0))
                logits = outs[x][2][:, :A].float().contiguous()
                pool[x] = states[x]
                if x < S - 1:
                    _lib.check(lib.hz_trees_backprop_traverse(
                        roots.handle, st, x, CONST["discount"], dec[N:].data_ptr(), dec[:N].data_ptr(), logits.data_ptr(), 1,
                        mmt.data_ptr(), CONST["delta"], CONST["pb_c_base"], CONST["pb_c_init"], ix.data_ptr(), None,
                        la.data_ptr(), None, pool.data_ptr(), hidden.data_ptr(), F * eb))
                    record()
                else:
                    _lib.check(lib.hz_trees_backprop(roots.handle, st, x, CONST["discount"], dec[N:].data_ptr(),
                                                     dec[:N].data_ptr(), logits.data_ptr(), 1, mmt.data_ptr()))
        v, val = roots.get_stats_tensors()
        e = roots.export(S)
        results.append(dict(trace=trace, visits=v.cpu(), values=val.cpu(), mm=mmt.cpu().clone(), ev=e["visits"].cpu(),
                            evs=e["value_sum"].cpu(), er=e["reward"].cpu(), plen=e["path_len"].cpu(), pool=pool.cpu(),
                            traj=roots.get_trajectories()))
    a, b = results
    assert len(a["trace"]) == len(b["trace"]) == S - 1
    for s, ((ix0, la0, b0), (ix1, la1, b1)) in enumerate(zip(a["trace"], b["trace"])):
        assert torch.equal(ix0, ix1) and torch.equal(la0, la1), f"traverse differs at simulation {s}"
        assert torch.equal(b0, b1), f"hand-off batch differs at simulation {s}"
    assert torch.equal(a["visits"], b["visits"]) and torch.equal(a["ev"], b["ev"]) and torch.equal(a["plen"], b["plen"])
    for k in ("values", "mm", "evs", "er"):
        assert bits_equal(a[k].numpy(), b[k].numpy()), k
    assert torch.equal(a["pool"], b["pool"]) and a["traj"] == b["traj"]
    assert (a["visits"].sum(1) == S - 1).all()
    return a


@pytest.mark.parametrize("N,A,S,width,dtype", [
    (300, 20, 30, 201, torch.float16),     # Hanabi-Full shapes, q in 2 registers per lane
    (129, 11, 40, 51, torch.float32),      # Hanabi-Small shapes, float pool
    (64, 20, 130, 201, torch.float16),     # capacity > 64: 8 q registers per lane
    (33, 20, 300, 201, torch.float32),     # capacity > 256: general back-propagation routine
    (2048, 20, 200, 201, torch.float16),   # BASELINE configs[4] per-GPU shard: 16384 trees x 200 sims over 8 GPUs
    (300, 20, 30, 21, torch.float16),      # narrow support: 3 of the decode's 32 lanes hold logits
    (129, 11, 40, 21, torch.float32),
    (300, 20, 30, 255, torch.float16),     # the widest odd support: every lane, the last one 7 columns
    (129, 11, 40, 255, torch.float32),
])
def test_search_step_equals_generic_calls(N, A, S, width, dtype):
    _run(N, A, S, width, dtype)


def test_search_step_deep_path_fallback():
    r = _run(24, 20, 60, 201, torch.float16, deep=True)
    assert int(r["plen"].max()) > 40           # the path outgrew one warp: general routine taken


def _search_step_vs_oracle(N, A, S, width, dtype, seed, tie=None, tree_offset=0, check_every=1, n_oracle=None, stage_limit=0):
    """The production launch (hz_trees_search_step, hidden state written straight into pool[x] as the search loop
    does) in lock-step with the CPU oracle: the oracle is fed hz_support_decode's values/rewards (the same
    arithmetic sequence as the fused decode) and the policy logits as float32.  Compares (ix, action) per
    simulation for every tree and visits / values / min-max / trajectories at the end, bit for bit.
    n_oracle: compare only the first n_oracle trees against the oracle (the oracle is scalar C)."""
    from hanabizero_b200 import _lib, cytree
    from oracle import loader as L
    lib = _lib.load()
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev).manual_seed(seed)
    F, OH = 512, 32 if A > 16 else 16
    P3 = (width + 7) // 8 * 8
    n_o = N if n_oracle is None else n_oracle
    d = tree_inputs(N, A, S, seed)
    support = (torch.arange(width, device=dev, dtype=torch.float32) - (width - 1) // 2)
    eb = torch.empty(0, dtype=dtype).element_size()
    st = torch.cuda.current_stream().cuda_stream
    roots = cytree.Roots(N, A, S)
    cpu = L.oracle_tree(n_o, A, S)
    if tie is not None:
        roots.set_tie_break("random", tie, tree_offset)
        cpu.set_tie(1, tie, tree_offset)
    roots.prepare(CONST["frac"], d["noise"], d["reward"], d["logits"], d["mask"])
    cpu.prepare(CONST["frac"], d["noise"][:n_o], d["reward"][:n_o], d["logits"][:n_o], d["mask"][:n_o])
    mm = cytree.MinMaxStatsList(N)
    mm.set_delta(CONST["delta"])
    mmt = mm.tensor(dev)
    pool = torch.zeros(S + 1, N, F, device=dev, dtype=dtype)
    pool[0] = torch.rand(N, F, device=dev, generator=gen).to(dtype)
    batch = torch.zeros(N, F + OH, device=dev, dtype=dtype)
    ix = torch.zeros(N, dtype=torch.int32, device=dev)
    la = torch.zeros(N, dtype=torch.int32, device=dev)
    cur = torch.zeros(3, N, P3, device=dev, dtype=dtype)
    dec = torch.zeros(2 * N, device=dev)
    io = _lib.SearchIO()
    io.value_logits, io.ld_value = cur[0].data_ptr(), P3
    io.reward_logits, io.ld_reward = cur[1].data_ptr(), P3
    io.policy_logits, io.ld_policy = cur[2].data_ptr(), P3
    io.next_state, io.ld_state = None, 0
    io.support, io.support_width, io.support_delta = support.data_ptr(), width, 1.0
    io.elem_bytes, io.sanitize_nan = eb, 1
    io.pool, io.state_cols = pool.data_ptr(), F
    io.out_batch, io.ld_batch, io.onehot_cols = batch.data_ptr(), F + OH, OH
    io.out_ix, io.out_action = ix.data_ptr(), la.data_ptr()
    io.minmax, io.value_delta_max = mmt.data_ptr(), CONST["delta"]
    io.discount, io.pb_c_base, io.pb_c_init = CONST["discount"], CONST["pb_c_base"], CONST["pb_c_init"]
    io.stage_limit = stage_limit
    ref = ctypes.byref(io)

    def compare(x):
        b = cpu.traverse(CONST["pb_c_base"], CONST["pb_c_init"], CONST["discount"])
        gi, ga = ix[:n_o].cpu().numpy(), la[:n_o].cpu().numpy()
        assert (gi == b[0]).all(), f"ix differs at simulation {x}: trees {np.flatnonzero(gi != b[0])[:8]}"
        assert (ga == b[2]).all(), f"action differs at simulation {x}: trees {np.flatnonzero(ga != b[2])[:8]}"
        rows = torch.arange(N, device=dev)
        assert torch.equal(batch[:, :F], pool[ix.long(), rows]), f"hand-off hidden rows at simulation {x}"
        onehot = torch.zeros(N, OH, device=dev, dtype=dtype)
        onehot[rows, la.long()] = 1.0
        assert torch.equal(batch[:, F:], onehot), f"hand-off one-hot at simulation {x}"

    _lib.check(lib.hz_trees_search_step(roots.handle, st, 0, 1, ref))
    compare(0)
    for x in range(1, S):
        cur.copy_(torch.randn(3, N, P3, device=dev, generator=gen).to(dtype))
        pool[x] = torch.rand(N, F, device=dev, generator=gen).to(dtype)   # what the dynamics GEMM would have written
        vr = cur[:2].reshape(2 * N, P3)
        _lib.check(lib.hz_support_decode(st, vr.data_ptr(), eb, support.data_ptr(), dec.data_ptr(), 2 * N, width, P3, 1.0))
        _lib.check(lib.hz_trees_search_step(roots.handle, st, x, 1 if x < S - 1 else 0, ref))
        h = dec.cpu().numpy()
        cpu.backprop(x, CONST["discount"], h[N:N + n_o], h[:n_o], cur[2][:n_o, :A].float().cpu().numpy())
        if x < S - 1 and (x % check_every == 0 or x > S - 4):
            compare(x)
        elif x < S - 1:
            cpu.traverse(CONST["pb_c_base"], CONST["pb_c_init"], CONST["discount"])
    v, val = roots.get_stats_tensors()
    ov, oval, omm = cpu.stats()
    assert (v[:n_o].cpu().numpy() == ov).all(), "visit counts"
    assert (v.sum(1) == S - 1).all()
    np.testing.assert_allclose(val[:n_o].cpu().numpy(), oval, rtol=1e-5, atol=0)      # north-star tolerance
    assert bits_equal(val[:n_o].cpu().numpy(), oval) and bits_equal(mmt[:n_o].cpu().numpy(), omm), "values / min-max bits"
    tr = roots.get_trajectories()
    otr = cpu.trajectories(S)
    for i in range(0, n_o, max(1, n_o // 64)):
        assert tr[i] == otr[i][otr[i] >= 0].tolist(), f"trajectory of tree {i}"
    return v.cpu().numpy()


@pytest.mark.parametrize("N,A,S,width,dtype,seed", [
    (200, 20, 50, 201, torch.float16, 11),    # fully staged in shared memory
    (37, 11, 50, 51, torch.float32, 12),      # Hanabi-Small shapes
    (5, 20, 16, 201, torch.float16, 13),      # capacity + 1 < 32 (path row padding), smoke()'s shape
    (4096, 20, 50, 201, torch.float16, 14),   # BASELINE configs[3] on one GPU: partially staged (one wave of CTAs)
    (2048, 20, 200, 201, torch.float16, 15),  # BASELINE configs[4] per-GPU shard
])
def test_search_step_lockstep_vs_oracle(N, A, S, width, dtype, seed):
    _search_step_vs_oracle(N, A, S, width, dtype, seed, check_every=1 if N < 1000 else 8)


@pytest.mark.parametrize("N,S,limit", [(200, 50, 4), (130, 50, 1), (2048, 200, 4)])
def test_search_step_with_a_staging_limit_vs_oracle(N, S, limit):
    """hz_search_io.stage_limit (the setting for several searches in flight: few nodes staged in shared memory, q read
    from global memory) must not change a single bit."""
    _search_step_vs_oracle(N, 20, S, 201, torch.float16, 21 + limit, check_every=1 if N < 1000 else 8, stage_limit=limit)


def test_search_step_random_tie_break_matches_oracle_and_shards():
    """Tie mode "random": same tie list as the reference, draws from the counter-based generator — bit-exact against
    the oracle running the same generator, and a shard with tree_offset draws what the full batch draws."""
    N, A, S = 96, 20, 30
    full = _search_step_vs_oracle(N, A, S, 201, torch.float16, 21, tie=1234)
    first = _search_step_vs_oracle(N, A, S, 201, torch.float16, 21)
    assert full.shape == first.shape    # (continuous random inputs: ties are rare, both runs are valid searches)


def test_support_width_over_256_is_rejected():
    from hanabizero_b200 import _lib, cytree
    lib = _lib.load()
    dev = torch.device("cuda")
    roots = cytree.Roots(4, 20, 8)
    roots.prepare_no_noise(np.zeros(4, np.float32), np.zeros((4, 20), np.float32), np.ones((4, 20), np.int32))
    mmt = cytree.MinMaxStatsList(4).tensor(dev)
    buf = torch.zeros(3, 4, 512, device=dev, dtype=torch.float16)
    pool = torch.zeros(9, 4, 512, device=dev, dtype=torch.float16)
    batch = torch.zeros(4, 544, device=dev, dtype=torch.float16)
    sup = torch.zeros(512, device=dev)
    io = _lib.SearchIO()
    io.value_logits, io.ld_value, io.reward_logits, io.ld_reward = buf[0].data_ptr(), 512, buf[1].data_ptr(), 512
    io.policy_logits, io.ld_policy = buf[2].data_ptr(), 512
    io.support, io.support_width, io.support_delta, io.elem_bytes = sup.data_ptr(), 300, 1.0, 2
    io.pool, io.state_cols, io.out_batch, io.ld_batch, io.onehot_cols = pool.data_ptr(), 512, batch.data_ptr(), 544, 32
    io.minmax, io.value_delta_max, io.discount, io.pb_c_base, io.pb_c_init = mmt.data_ptr(), 0.006, 0.999, 19652, 1.25
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.hz_trees_search_step(roots.handle, st, 0, 1, ctypes.byref(io)))
    assert lib.hz_trees_search_step(roots.handle, st, 1, 1, ctypes.byref(io)) == _lib.HZ_ERR_ARG
