"""GPU: the reanalyze pipeline.  hz_obs_pack_windows against hz_obs_pack of the windows expanded by torch, byte for
byte, over layouts, frame formats, stacks, positions, x types, row strides, sources and wave fills; hz_wave_policy against
hz_visit_policy, bit for bit; ReanalyzePipeline's targets against the explicit chain (submit_observations of the
expanded stacks, then hz_visit_policy), bit for bit, with garbage frames past the end of episodes; against
reanalyze_policies on real positions; and asynchronous use with a weight update."""
import ctypes

import numpy as np
import pytest
import torch

from test_search_obs_gpu import LAYOUTS, _frames, _layout, _legal, _mask_words, _model, _strings, _with_row_stride

pytestmark = pytest.mark.gpu


def _expand(windows, S, P):
    """[rows, S + P - 1, ...] windows -> [rows * P, S, ...] stacks: stack p of window i = frames p .. p + S - 1."""
    rows = windows.shape[0]
    return torch.stack([windows[:, p:p + S] for p in range(P)], 1).reshape(rows * P, S, *windows.shape[2:])


def _pin(t):
    """The same values in page-locked host memory, row stride kept."""
    return torch.empty_strided(t.shape, t.stride(), dtype=t.dtype, pin_memory=True).copy_(t)


SOURCES = [(f, where) for where in ("device", "pinned") for f in ("f32", "u8", "bits")]


@pytest.mark.parametrize("elem", ["half", "float"])
@pytest.mark.parametrize("P", [1, 2, 6])
@pytest.mark.parametrize("S", [1, 4])
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_window_pack_equals_the_expanded_pack(layout, S, P, elem):
    """Waves of 4 full and partial (3 of 4), tickets cycling through F32 / U8 / BITS windows from the device and from
    pinned host memory, window rows longer than the window, legal moves in the three formats, with and without noise:
    x, legal and noise staging of hz_obs_pack_windows equal hz_obs_pack over the torch-expanded stacks byte for byte,
    and the padding rows are zero."""
    from hanabizero_b200 import _lib
    lib = _lib.load()
    full, D, stride, A, W, off, gdim = _layout(layout)
    dtype = torch.float16 if elem == "half" else torch.float32
    G, rows = 4, 13
    n = rows * P
    L = _lib.ObsLayout(stack=S, frame_dim=D, frame_stride=stride, elem_bytes=dtype.itemsize, frame_words=W, bit_offset=off)
    st = torch.cuda.current_stream().cuda_stream
    rotation = (S + 3 * P + (elem == "half")) % len(SOURCES)
    for count in (G, 3):
        outs = []
        for windows in (True, False):
            x = torch.full((G * n, S * stride), -1, dtype=dtype, device="cuda")
            legal_out = torch.full((G * n, A), -1, dtype=torch.int32, device="cuda")
            noise_out = torch.full((G * n, A), -1.0, device="cuda")
            table, keep = [], []
            for k in range(count):
                seed = 10 * count + k
                fmt, where = SOURCES[(rotation + k) % len(SOURCES)]
                frames = _frames(rows, S + P - 1, D, seed)
                if fmt == "f32":
                    src, code = frames.float(), _lib.HZ_OBS_F32
                elif fmt == "u8":
                    src, code = frames, _lib.HZ_OBS_U8
                else:
                    src, code = _strings(frames, off, gdim, seed), _lib.HZ_OBS_BITS
                src = src if windows else _expand(src, S, P)
                src = _with_row_stride(src, 1 + 16 * (k % 2))                 # rows longer than the window or stack
                legal = _legal(n, A, seed)
                leg, lcode = [(legal, _lib.HZ_LEGAL_I32), (_with_row_stride(legal.float(), 3), _lib.HZ_LEGAL_F32),
                              (_mask_words(legal)[:, 0], _lib.HZ_LEGAL_MASK)][k % 3]
                noise = None if k == 1 else torch.rand(n, A, device="cuda", generator=torch.Generator(
                    device="cuda").manual_seed(seed))
                if where == "pinned":
                    src, leg, noise = _pin(src), _pin(leg), None if noise is None else _pin(noise)
                keep.append((src, leg, noise))
                table.append(_lib.ObsTicket(obs=src.data_ptr(), ld_obs=src.stride(0), legal=leg.data_ptr(),
                                            ld_legal=leg.stride(0), noise=None if noise is None else noise.data_ptr(),
                                            obs_format=code, legal_format=lcode))
            tab = (_lib.ObsTicket * count)(*table)
            if windows:
                rc = lib.hz_obs_pack_windows(st, 0, tab, count, G, n, A, ctypes.byref(L), P, x.data_ptr(),
                                             legal_out.data_ptr(), noise_out.data_ptr())
            else:
                rc = lib.hz_obs_pack(st, 0, tab, count, G, n, A, ctypes.byref(L), x.data_ptr(), legal_out.data_ptr(),
                                     noise_out.data_ptr())
            _lib.check(rc)
            torch.cuda.synchronize()
            outs.append((x, legal_out, noise_out))
        (xw, lw, nw), (xs, ls, ns) = outs
        assert torch.equal(xw.view(torch.int16 if elem == "half" else torch.int32),
                           xs.view(torch.int16 if elem == "half" else torch.int32)), (count, "x")
        assert torch.equal(lw, ls) and torch.equal(nw.view(torch.int32), ns.view(torch.int32)), count
        pad = slice(count * n, G * n)
        assert not xw[pad].any() and not lw[pad].any() and not nw[pad].any(), count
        assert xw[:count * n].any(), count


@pytest.mark.parametrize("n", [1, 37, 300])
def test_wave_policy_equals_visit_policy(n):
    """Random visit counts (zero rows among the masked-out ones) in a wave's statistics buffer; full and partial waves,
    tickets with and without a mask (device and pinned), outputs in device and in pinned host memory: float64 targets
    equal hz_visit_policy of each ticket's rows bit for bit."""
    from hanabizero_b200 import _lib
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    for A in (20, 11):
        G = 5
        g = torch.Generator(device="cuda").manual_seed(n * A)
        visits = torch.randint(0, 60, (G * n, A), device="cuda", generator=g, dtype=torch.int32)
        visits[:, 0] += 1
        masks = (torch.rand(G * n, device="cuda", generator=g) < 0.7).to(torch.uint8)
        visits[masks == 0] *= (torch.rand(G * n, device="cuda", generator=g) < 0.5).int()[masks == 0].unsqueeze(1)
        stats = torch.cat([visits.view(-1), torch.randint(0, 1 << 30, (G * n,), device="cuda", dtype=torch.int32)])
        for count in (G, 2):
            table, outs, want = [], [], []
            for k in range(count):
                rows = slice(k * n, (k + 1) * n)
                mask = None if k % 2 else masks[rows].clone()
                if k % 3 == 1:
                    mask = _pin(mask) if mask is not None else None
                out = torch.full((n, A), -7.0, dtype=torch.float64, device="cuda")
                if k % 2 == 0 and k > 0:
                    out = _pin(out)
                ref = torch.empty(n, A, dtype=torch.float64, device="cuda")
                m = None if mask is None else mask.cuda()
                _lib.check(lib.hz_visit_policy(st, visits[rows].contiguous().data_ptr(),
                                               None if m is None else m.data_ptr(), n, A, ref.data_ptr(), None))
                outs.append((out, mask))
                want.append(ref)
                table.append(_lib.PolicyTicket(mask=None if mask is None else mask.data_ptr(), out=out.data_ptr()))
            _lib.check(lib.hz_wave_policy(st, 0, (_lib.PolicyTicket * count)(*table), count, G, n, A, stats.data_ptr()))
            torch.cuda.synchronize()
            for k, ((out, _), ref) in enumerate(zip(outs, want)):
                assert torch.equal(out.cuda().view(torch.int64), ref.view(torch.int64)), (A, count, k)


# ---- the pipeline ---------------------------------------------------------------------------------------------------

def _cfg(A, sims=12):
    from hanabizero_b200.mcts import SearchConfig
    cfg = SearchConfig(num_simulations=sims, amp_type="torch_amp")
    cfg.action_space_size = A
    return cfg


def _sample(batch, K, S, D, A, seed, ends=True):
    """Trajectory windows of one reanalyze ticket: frames [batch, K + S, D], legal [batch, K + 1, A], mask
    [batch, K + 1].  With `ends`, sample b's episode ends after position e_b - 1 (e_b in 1..K + 1): later positions are
    masked out with all-zero legal rows, and window frames from e_b + S - 1 on are random garbage."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    frames = (torch.rand(batch, K + S, D, device="cuda", generator=g) < 0.3).to(torch.uint8)
    legal = (torch.rand(batch, K + 1, A, device="cuda", generator=g) < 0.5).int()
    legal[:, :, seed % A] = 1
    mask = torch.ones(batch, K + 1, dtype=torch.uint8, device="cuda")
    garbage = torch.zeros(batch, K + S, dtype=torch.bool, device="cuda")
    if ends:
        e = torch.randint(1, K + 2, (batch,), device="cuda", generator=g)
        pos = torch.arange(K + 1, device="cuda")
        mask = (pos < e.unsqueeze(1)).to(torch.uint8)
        legal *= mask.unsqueeze(2).int()
        garbage = torch.arange(K + S, device="cuda") >= (e + S - 1).unsqueeze(1)
    return dict(frames=frames, legal=legal, mask=mask, garbage=garbage)


def _windows(t, fmt, seed, off=0, gdim=None):
    """The sample's windows in a frame format, garbage frames filled with noise of that format."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    frames, bad = t["frames"], t["garbage"]
    if fmt == "u8":
        w = frames.clone()
        w[bad] = torch.randint(0, 256, (int(bad.sum()), frames.shape[2]), device="cuda", generator=g, dtype=torch.uint8)
    elif fmt == "f32":
        w = frames.float()
        w[bad] = torch.randn(int(bad.sum()), frames.shape[2], device="cuda", generator=g) * 100
    else:
        w = _strings(frames, off, gdim, seed)
        w[bad] = torch.randint(-2 ** 31, 2 ** 31 - 1, (int(bad.sum()), w.shape[2]), device="cuda", generator=g,
                               dtype=torch.int32)
    return w


def _chain(ref_pipe, windows, legal, mask, noise, S, P, fraction):
    """The explicit chain: submit_observations of the torch-expanded stacks, then hz_visit_policy with the mask."""
    from hanabizero_b200 import _lib
    n, A = ref_pipe.n, ref_pipe.a
    visits = torch.empty(n, A, dtype=torch.int32, device="cuda")
    t = ref_pipe.submit_observations(fraction, noise, _expand(windows, S, P).contiguous(), legal.reshape(n, A),
                                     visits)
    ref_pipe.wait(t)
    out = torch.empty(n, A, dtype=torch.float64, device="cuda")
    _lib.check(_lib.load().hz_visit_policy(torch.cuda.current_stream().cuda_stream, visits.data_ptr(),
                                           mask.reshape(n).contiguous().data_ptr(), n, A, out.data_ptr(), None))
    torch.cuda.synchronize()
    return out


def _noise(cfg, roots, A, legal, seed, step):
    from hanabizero_b200.selfplay import dirichlet_noise
    return dirichlet_noise(roots, A, cfg.root_dirichlet_alpha, "cuda", seed, step) * legal.reshape(roots, A).float()


def test_pipeline_targets_equal_the_explicit_chain():
    """ReanalyzePipeline (K = 5, positions 6, waves of 3 tickets, a partial last wave) with u8, f32 and bit windows and
    both legal forms: every target equals the explicit chain over the expanded stacks bit for bit.  Masked positions with
    garbage frames and all-zero legal rows give zero rows, and other garbage gives the same targets."""
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    from hanabizero_b200.reanalyze import ReanalyzePipeline
    full, D, _, A, W, off, gdim = _layout("full-global")
    batch, K, S, G = 32, 5, 4, 3
    cfg = _cfg(A)
    model = _model(full, D, S, A)
    rp = ReanalyzePipeline(cfg, model, batch, K, S, depth=2, wave=G)
    assert rp.pipe.executor == "rows"
    ref = SearchPipeline(MCTS(cfg), model, batch * (K + 1), A, depth=2, wave=G, executor="rows", stack=S)
    samples, ids = [], []
    for k in range(5):
        fmt = ("u8", "f32", "bits")[k % 3]
        t = _sample(batch, K, S, D, A, seed=20 + k)
        win = _windows(t, fmt, seed=30 + k, off=off, gdim=gdim)
        legal = _mask_words(t["legal"].view(-1, A))[:, 0].view(batch, K + 1) if k % 2 else t["legal"]
        out = torch.full((batch, K + 1, A), -1.0, dtype=torch.float64, device="cuda")
        ids.append(rp.submit(win, legal, t["mask"], noise_seed=5, noise_step=k, out=out))
        samples.append((t, win, fmt))
    rp.drain()
    torch.cuda.synchronize()
    for k, ((t, win, fmt), tid) in enumerate(zip(samples, ids)):
        got = rp.result(tid)
        noise = _noise(cfg, batch * (K + 1), A, t["legal"], 5, k)
        want = _chain(ref, win, t["legal"], t["mask"], noise, S, K + 1, cfg.root_exploration_fraction)
        assert torch.equal(got.reshape(-1, A).view(torch.int64), want.view(torch.int64)), (k, fmt)
        m = t["mask"].reshape(-1).bool()
        assert not got.reshape(-1, A)[~m].any() and bool(m.any()) and bool((~m).any()), k
        sums = got.reshape(-1, A)[m].sum(1)
        assert float((sums - 1).abs().max()) < 1e-12, k
    # other garbage past the episode ends: the same targets
    t, win, fmt = samples[0]
    other = _windows(t, fmt, seed=99)
    assert not torch.equal(other, win)
    tid = rp.submit(other, t["legal"], t["mask"], noise_seed=5, noise_step=0)
    assert torch.equal(rp.result(tid).view(torch.int64), rp.result(ids[0]).view(torch.int64))


def _trajectories(batch, steps, seed):
    """Real Hanabi-Full play: batch games, 6 random moves, then `steps` recorded moves -> global frames float
    [batch, steps, 785] and legal masks float [batch, steps, A] (legal of the position each frame shows)."""
    from hanabizero_b200.hanabi_env import HanabiVecEnv
    env = HanabiVecEnv(batch, "Hanabi-Full", np.arange(batch) + seed)
    g, _, legal = env.reset_all()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    frames, legals = [], []
    for i in range(6 + steps):
        if i >= 6:
            frames.append(g.clone())
            legals.append(legal.clone())
        g, _, legal, _, _, _ = env.step_all(torch.multinomial(legal, 1, generator=gen).view(-1).int(), auto_reset=True)
    env.check()
    return torch.stack(frames, 1), torch.stack(legals, 1)


def test_targets_agree_with_reanalyze_policies(record_property):
    """1536 real Hanabi-Full positions (256 windows, K = 5, stack 4, 50 simulations, fp16), noise from the same
    (noise_seed, noise_step): masked-out rows are zero in both, every kept row sums to 1 within 1e-12, and the arg-max
    of at least 99 % of the kept rows agrees (InitialPlan rounds the root inference differently from the module)."""
    from hanabizero_b200.reanalyze import ReanalyzePipeline, reanalyze_policies
    batch, K, S, A, D = 256, 5, 4, 20, 785
    frames, legal = _trajectories(batch, K + S, seed=3)
    legal = legal[:, S - 1:].clone()                       # position p shows frame p + S - 1
    mask = torch.ones(batch, K + 1, dtype=torch.uint8, device="cuda")
    mask[::7, 4:] = 0
    legal[mask == 0] = 0
    cfg = _cfg(A, sims=50)
    model = _model(True, D, S, A)
    rp = ReanalyzePipeline(cfg, model, batch, K, S, depth=2)
    got = rp.result(rp.submit(frames.to(torch.uint8), legal, mask, noise_seed=9, noise_step=4)).reshape(-1, A)
    stacks = _expand(frames, S, K + 1).reshape(batch * (K + 1), S * D)
    want = reanalyze_policies(cfg, model, stacks, legal.reshape(-1, A), mask.reshape(-1), K, as_tensor=True,
                              noise_seed=9, noise_step=4).reshape(-1, A)
    m = mask.reshape(-1).bool()
    assert not got[~m].any() and not want[~m].any()
    assert float((got[m].sum(1) - 1).abs().max()) < 1e-12 and float((want[m].sum(1) - 1).abs().max()) < 1e-12
    agree = float((got[m].argmax(1) == want[m].argmax(1)).double().mean())
    record_property("agreement", f"{agree:.4f}")
    assert agree >= 0.99, agree


def test_asynchronous_tickets_and_a_weight_update():
    """Six tickets submitted ahead of their results (pinned host and device inputs mixed, waves of 2, 3 slots) each equal
    the same ticket submitted alone to a fresh pipeline; after drain() and a weight update the next ticket equals a fresh
    pipeline on the updated module and differs from the same ticket before the update."""
    from hanabizero_b200.reanalyze import ReanalyzePipeline
    full, D, _, A, _, _, _ = _layout("small-local")
    batch, K, S = 24, 3, 4
    cfg = _cfg(A)
    model = _model(full, D, S, A, seed=1)
    make = lambda: ReanalyzePipeline(cfg, model, batch, K, S, mdp="local", depth=3, wave=2)
    rp = make()
    inputs = []
    for k in range(6):
        t = _sample(batch, K, S, D, A, seed=50 + k)
        win, legal, mask = _windows(t, "u8", seed=60 + k), t["legal"], t["mask"]
        if k % 2:
            win, legal, mask = _pin(win.cpu()), _pin(legal.cpu()), _pin(mask.cpu())
        inputs.append((win, legal, mask, k))
    outs = [_pin(torch.empty(batch, K + 1, A, dtype=torch.float64)) if k % 3 == 2 else None for k in range(6)]
    ids = [rp.submit(w, l, m, noise_seed=1, noise_step=s, out=o) for (w, l, m, s), o in zip(inputs, outs)]
    got = [rp.result(t).clone() for t in ids]
    alone = []
    for w, l, m, s in inputs:
        fresh = make()
        alone.append(fresh.result(fresh.submit(w, l, m, noise_seed=1, noise_step=s)))
    for k, (a, b) in enumerate(zip(got, alone)):
        assert torch.equal(a.cuda().view(torch.int64), b.view(torch.int64)), k
    rp.drain()
    model.load_state_dict(_model(full, D, S, A, seed=2).state_dict())
    w, l, m, s = inputs[0]
    after = rp.result(rp.submit(w, l, m, noise_seed=1, noise_step=s))
    fresh = make()
    assert torch.equal(after.view(torch.int64), fresh.result(fresh.submit(w, l, m, noise_seed=1,
                                                                          noise_step=s)).view(torch.int64))
    assert not torch.equal(after, got[0].cuda())
