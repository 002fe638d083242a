"""GPU: observation tickets (SearchPipeline.submit_observations, hz_obs_pack).  The pack kernel against torch, exactly,
for every frame and legal format, layout, stack, input type, row count, wave fill and source memory; the pipeline's
results against an explicit chain over the same wave (torch-built input -> InitialPlan -> prepare -> run_multi), bit for
bit; format independence; the root inference against the float64 module; kinds of tickets in one pipeline; weight
updates; and a closed host-driven actor loop on EnvPipeline(fmt="bits")."""
import ctypes

import numpy as np
import pytest
import torch

from test_initial_plan_gpu import LAYOUTS, _assert_within, _float64, _net, _ratios, _reference

pytestmark = pytest.mark.gpu

GAME = {True: "Hanabi-Full", False: "Hanabi-Small"}
BIT_OFFSET = {"full-global": 0, "full-local": 125, "small-global": 0, "small-local": 20}


def _layout(name):
    """(full, D, frame_stride, A, W, bit_offset, global_dim), the frame's place in the packed string read from the env."""
    from hanabizero_b200.hanabi_env import HanabiVecEnv, frame_layout
    full, D, stride, A, _ = LAYOUTS[name]
    dim, W, off = frame_layout(GAME[full], name.split("-")[1])
    assert (dim, off) == (D, BIT_OFFSET[name])
    return full, D, stride, A, W, off, HanabiVecEnv(1, GAME[full]).global_dim


def _strings(frames, off, global_dim, seed):
    """0/1 frames [n, S, D] -> packed strings int32 [n, S, W]: the frame at bits [off, off + D), random bits before it
    (the own-hand prefix of a local view), zeros after global_dim."""
    n, S, D = frames.shape
    g = torch.Generator(device="cuda").manual_seed(seed)
    full = (torch.rand(n, S, global_dim, device="cuda", generator=g) < 0.5).to(torch.uint8)
    full[:, :, off:off + D] = frames
    W = (global_dim + 31) // 32
    bits = np.zeros((n, S, 32 * W), np.uint8)
    bits[:, :, :global_dim] = full.cpu().numpy()
    packed = np.packbits(bits, axis=2, bitorder="little").view(np.int32)
    return torch.from_numpy(packed.copy()).cuda()


def _frames(n, S, D, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.rand(n, S, D, device="cuda", generator=g) < 0.3).to(torch.uint8)


def _legal(n, A, seed):
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    legal = (torch.rand(n, A, device="cuda", generator=g) < 0.5).int()
    legal[:, seed % A] = 1
    return legal


def _mask_words(legal):
    """int32 meta rows [n, 4] with the legal bit mask in word 0 (EnvPipeline's layout)."""
    n, A = legal.shape
    words = (legal.long() << torch.arange(A, device=legal.device)).sum(1)
    meta = torch.zeros(n, 4, dtype=torch.int32, device=legal.device)
    meta[:, 0] = words.to(torch.int32)
    meta[:, 1:] = 7
    return meta


def _with_row_stride(t, extra):
    """The same values in a buffer whose rows are `extra` elements longer (a row stride the kernel must follow)."""
    n = t.shape[0]
    flat = t.reshape(n, -1)
    buf = torch.full((n, flat.shape[1] + extra), 3, dtype=t.dtype, device=t.device)
    buf[:, :flat.shape[1]] = flat
    return buf[:, :flat.shape[1]].view(t.shape)


def _ticket_inputs(fmt, legal_fmt, frames, legal, off, global_dim, seed, pinned):
    """(ObsTicket fields, tensors kept alive) of one ticket in the given formats."""
    from hanabizero_b200 import _lib
    n, S, D = frames.shape
    if fmt == "f32":
        obs, code = _with_row_stride(frames.float(), 3), _lib.HZ_OBS_F32          # rows not 16-byte aligned
    elif fmt == "u8":
        obs, code = _with_row_stride(frames, 16 * (seed % 2)), _lib.HZ_OBS_U8
    else:
        obs, code = _with_row_stride(_strings(frames, off, global_dim, seed), seed % 3), _lib.HZ_OBS_BITS
    if legal_fmt == "i32":
        leg, lcode = legal, _lib.HZ_LEGAL_I32
    elif legal_fmt == "f32":
        leg, lcode = _with_row_stride(legal.float(), 5), _lib.HZ_LEGAL_F32
    else:
        leg, lcode = _mask_words(legal)[:, 0], _lib.HZ_LEGAL_MASK
    noise = None if seed % 4 == 3 else torch.rand(n, legal.shape[1], device="cuda")
    if pinned:
        # pin the whole underlying buffer and keep the row stride
        pin = lambda t: None if t is None else torch.empty_strided(t.shape, t.stride(), dtype=t.dtype,
                                                                   pin_memory=True).copy_(t)
        obs, leg, noise = pin(obs), pin(leg), pin(noise)
    t = _lib.ObsTicket(obs=obs.data_ptr(), ld_obs=obs.stride(0), legal=leg.data_ptr(), ld_legal=leg.stride(0),
                       noise=None if noise is None else noise.data_ptr(), obs_format=code, legal_format=lcode)
    return t, (obs, leg, noise)


FORMATS = [(f, l, p) for p in (False, True) for f in ("f32", "u8", "bits") for l in ("i32", "f32", "mask")]


@pytest.mark.parametrize("n", [1, 77, 512])
@pytest.mark.parametrize("elem", ["half", "float"])
@pytest.mark.parametrize("S", [1, 3, 4])
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_obs_pack_equals_torch(layout, S, elem, n):
    """Full waves of 8 and partial waves (3 of 8) whose tickets cycle through every frame format x legal format x
    device / pinned-host source; tickets with and without noise.  x, legal and noise staging equal torch's construction
    exactly; padding columns and padding rows are zero."""
    from hanabizero_b200 import _lib
    lib = _lib.load()
    full, D, stride, A, W, off, gdim = _layout(layout)
    dtype = torch.float16 if elem == "half" else torch.float32
    G = 8
    L = _lib.ObsLayout(stack=S, frame_dim=D, frame_stride=stride, elem_bytes=dtype.itemsize, frame_words=W, bit_offset=off)
    rotation = (S * 7 + n + (elem == "half")) % len(FORMATS)
    for count in (G, 3):
        x = torch.full((G * n, S * stride), -1, dtype=dtype, device="cuda")
        legal_out = torch.full((G * n, A), -1, dtype=torch.int32, device="cuda")
        noise_out = torch.full((G * n, A), -1.0, device="cuda")
        want_x, want_legal, want_noise = torch.zeros_like(x), torch.zeros_like(legal_out), torch.zeros_like(noise_out)
        table, keep = [], []
        for k in range(count):
            seed = 100 * count + k
            fmt, lfmt, pinned = FORMATS[(rotation + k) % len(FORMATS)]
            frames, legal = _frames(n, S, D, seed), _legal(n, A, seed)
            t, held = _ticket_inputs(fmt, lfmt, frames, legal, off, gdim, seed, pinned)
            table.append(t)
            keep.append(held)
            rows = slice(k * n, (k + 1) * n)
            want_x[rows].view(n, S, stride)[:, :, :D] = frames.to(dtype)
            want_legal[rows] = legal
            if held[2] is not None:
                want_noise[rows] = held[2].cuda()
        tab = (_lib.ObsTicket * count)(*table)
        _lib.check(lib.hz_obs_pack(torch.cuda.current_stream().cuda_stream, 0, tab, count, G, n, A, ctypes.byref(L),
                                   x.data_ptr(), legal_out.data_ptr(), noise_out.data_ptr()))
        torch.cuda.synchronize()
        assert torch.equal(x, want_x), (count, "x")
        assert torch.equal(legal_out, want_legal), (count, "legal")
        assert torch.equal(noise_out, want_noise), (count, "noise")
        # a wave without noise leaves the noise staging alone
        noise_out.fill_(-2.0)
        _lib.check(lib.hz_obs_pack(torch.cuda.current_stream().cuda_stream, 0, tab, count, G, n, A, ctypes.byref(L),
                                   x.data_ptr(), legal_out.data_ptr(), None))
        torch.cuda.synchronize()
        assert torch.equal(x, want_x) and bool((noise_out == -2.0).all())


def test_obs_pack_rejects_bad_pointers_without_launching():
    from hanabizero_b200 import _lib
    lib = _lib.load()
    n, A, S, D = 64, 20, 4, 785
    L = _lib.ObsLayout(stack=S, frame_dim=D, frame_stride=800, elem_bytes=2, frame_words=25, bit_offset=0)
    x = torch.zeros(n, S * 800, dtype=torch.float16, device="cuda")
    legal = torch.zeros(n, A, dtype=torch.int32, device="cuda")
    obs = torch.zeros(n, S * D, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def pack(obs_ptr=obs.data_ptr(), x_ptr=x.data_ptr(), fmt=_lib.HZ_OBS_F32):
        t = _lib.ObsTicket(obs=obs_ptr, ld_obs=S * D, legal=legal.data_ptr(), ld_legal=A, noise=None, obs_format=fmt,
                           legal_format=_lib.HZ_LEGAL_I32)
        return lib.hz_obs_pack(st, 0, (_lib.ObsTicket * 1)(t), 1, 1, n, A, ctypes.byref(L), x_ptr, legal.data_ptr(), None)

    assert pack() == _lib.HZ_OK
    torch.cuda.synchronize()
    before = lib.hz_launch_count()
    pageable = torch.zeros(n, S * D)
    assert pack(obs_ptr=pageable.data_ptr()) == _lib.HZ_ERR_ARG and b"page-locked" in lib.hz_last_error()
    assert pack(obs_ptr=obs.data_ptr() + 2) == _lib.HZ_ERR_ARG and b"aligned" in lib.hz_last_error()
    assert pack(x_ptr=x.data_ptr() + 8) == _lib.HZ_ERR_ARG and b"aligned" in lib.hz_last_error()
    assert lib.hz_launch_count() == before
    assert pack(obs_ptr=obs.data_ptr() + 1, fmt=_lib.HZ_OBS_U8) == _lib.HZ_OK     # bytes need no alignment
    torch.cuda.synchronize()


# ---- the pipeline ---------------------------------------------------------------------------------------------------

SIMS = 12


def _cfg(amp, sims=SIMS):
    from hanabizero_b200.mcts import SearchConfig
    return SearchConfig(num_simulations=sims, amp_type=amp)


def _model(full, D, S, A, seed=0):
    from hanabizero_b200.model import MuZeroNet, MuZeroNetFull
    torch.manual_seed(seed)
    return (MuZeroNetFull if full else MuZeroNet)(D * S, A).randomize_heads(std=0.05, seed=seed).to("cuda").eval()


def _obs_ticket(n, S, D, A, seed, noisy=True):
    frames = _frames(n, S, D, seed)
    return dict(frames=frames, legal=_legal(n, A, seed),
                noise=torch.rand(n, A, device="cuda") if noisy else None,
                visits=torch.full((n, A), -1, dtype=torch.int32, device="cuda"),
                values=torch.full((n,), float("nan"), device="cuda"))


def _submit_obs(pipe, t, obs=None, legal=None, fraction=0.25):
    return pipe.submit_observations(fraction, t["noise"], t["frames"].float() if obs is None else obs,
                                    t["legal"] if legal is None else legal, t["visits"], t["values"])


def _explicit_wave(pipe, mcts, tickets, fraction=0.25, owner=None):
    """The wave's search done by hand: torch-built x in InitialPlan.bound(G*n) -> run_bound -> prepare -> run_multi with
    the pipeline's executor, SM target and stage limit.  -> (visits, values) of the G*n trees."""
    from hanabizero_b200 import _lib, cytree
    plan, G, n, A, S = pipe._iplan, pipe.wave, pipe.n, pipe.a, pipe.stack
    b = plan.bound(G * n, owner=owner)
    if pipe.gemm_sm_target:
        _lib.check(plan.lib.hz_gemm_plan_set_sm_target(b.handle, pipe.gemm_sm_target))
    b.x.zero_()
    legal = torch.zeros(G * n, A, dtype=torch.int32, device="cuda")
    noise = torch.zeros(G * n, A, device="cuda")
    for k, t in enumerate(tickets):
        b.x[k * n:(k + 1) * n].view(n, S, plan.frame_stride)[:, :, :pipe.frame_dim] = t["frames"].to(plan.dtype)
        legal[k * n:(k + 1) * n] = t["legal"]
        if t["noise"] is not None:
            noise[k * n:(k + 1) * n] = t["noise"]
    logits = torch.empty(G * n, A, device="cuda")
    hidden = plan.run_bound(b, logits)
    roots = cytree.Roots(G * n, A, mcts.config.num_simulations)
    zeros = torch.zeros(G * n, device="cuda")
    if tickets[0]["noise"] is None:
        roots.prepare_no_noise(zeros, logits, legal)
    else:
        roots.prepare(fraction, noise, zeros, logits, legal)
    mcts.run_multi(roots, pipe.model, hidden, gemm_sm_target=pipe.gemm_sm_target, stage_limit=pipe.stage_limit,
                   executor=pipe.executor)
    return roots.get_stats_tensors()


def _assert_rows(t, visits, values, k, n, what=""):
    rows = slice(k * n, (k + 1) * n)
    assert torch.equal(t["visits"], visits[rows]), what
    assert torch.equal(t["values"].view(torch.int32), values[rows].view(torch.int32)), what


class _Owner:
    pass


@pytest.mark.parametrize("amp", ["torch_amp", "none"])
@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("executor", ["rows", "library"])
def test_observation_waves_equal_the_explicit_chain(executor, layout, amp):
    """Three waves per slot (eager search, capture, replays), the last without noise; frames in float32 from the device.
    fp32 plans have no row-block executor: they run the library chain whatever `executor` says."""
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    full, D, _, A, _, _, _ = _layout(layout)
    S, n, G, depth = 4, 128, 4, 2
    model = _model(full, D, S, A)
    pipe = SearchPipeline(MCTS(_cfg(amp)), model, n, A, depth=depth, executor=executor, wave=G, stack=S,
                          mdp=layout.split("-")[1])
    waves = [[_obs_ticket(n, S, D, A, 10 * w + p, noisy=w < 2 * depth) for p in range(G)] for w in range(3 * depth)]
    for wave in waves:
        for t in wave:
            _submit_obs(pipe, t)
    pipe.drain()
    torch.cuda.synchronize()
    ref, owner = MCTS(_cfg(amp)), _Owner()
    for w, wave in enumerate(waves):
        visits, values = _explicit_wave(pipe, ref, wave, owner=owner)
        for k, t in enumerate(wave):
            _assert_rows(t, visits, values, k, n, (w, k))
            assert int(t["visits"].sum()) == n * (SIMS - 1)


def test_formats_and_sources_give_identical_searches():
    """The same observations as float32, bytes and packed bits, with int32 / float / bit-mask legal moves, from the device
    and from pinned host memory, and pageable (the torch slow path): identical visits and values (waves of one)."""
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    full, D, _, A, W, off, gdim = _layout("full-local")
    S, n = 3, 200
    model = _model(full, D, S, A)
    pipe = SearchPipeline(MCTS(_cfg("torch_amp")), model, n, A, depth=2, executor="rows", stack=S, mdp="local")
    base = _obs_ticket(n, S, D, A, seed=5)
    strings = _strings(base["frames"], off, gdim, seed=5)
    forms = [("f32", base["frames"].float(), base["legal"]), ("u8", base["frames"], base["legal"].float()),
             ("bits", strings, _mask_words(base["legal"])[:, 0]), ("bits-2d", strings.view(n, S * W), base["legal"])]
    results = []
    for name, obs, legal in forms:
        for where in ("device", "pinned", "pageable"):
            o, l = obs, legal
            if where == "pinned":
                o, l = obs.cpu().pin_memory(), legal.cpu().pin_memory()
            elif where == "pageable":
                o, l = obs.cpu(), legal.cpu()
            t = dict(base, visits=torch.full((n, A), -1, dtype=torch.int32, device="cuda"),
                     values=torch.full((n,), float("nan"), device="cuda"))
            tid = _submit_obs(pipe, t, obs=o, legal=l)
            pipe.wait(tid)
            results.append(((name, where), t))
    torch.cuda.synchronize()
    first = results[0][1]
    assert int(first["visits"].sum()) == n * (SIMS - 1)
    for what, t in results[1:]:
        assert torch.equal(t["visits"], first["visits"]), what
        assert torch.equal(t["values"].view(torch.int32), first["values"].view(torch.int32)), what


@pytest.mark.parametrize("amp", ["torch_amp", "none"])
@pytest.mark.parametrize("layout", ["full-global", "small-local"])
def test_root_inference_matches_the_float64_module(layout, amp, record_property):
    """The slot's root inference buffers after an observation wave (a partial one: 3 of 4 tickets) are within the
    float64-module bounds of tests/test_initial_plan_gpu.py for the real rows."""
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    full, D, _, A, _, _, _ = _layout(layout)
    S, n, G = 4, 100, 4
    net = _net(full, D * S, A, 201 if full else 51, seed=3)
    net64 = _float64(net)
    pipe = SearchPipeline(MCTS(_cfg(amp)), net, n, A, depth=2, wave=G, stack=S, mdp=layout.split("-")[1])
    tickets = [_obs_ticket(n, S, D, A, seed=40 + k) for k in range(3)]
    ids = [_submit_obs(pipe, t, obs=t["frames"]) for t in tickets]
    pipe.wait(ids[0])
    torch.cuda.synchronize()
    b = pipe.slots[pipe._waves.slot_of(ids[0])]["ibound"]
    ref = _reference(net64, torch.cat([t["frames"].view(n, -1) for t in tickets]))

    class Rows:          # the real rows of the bound's buffers
        pass
    rows = Rows()
    for k in ("x", "state", "h1", "out", "r1", "t1") + (("r2", "r3", "t2", "xb") if full else ()):
        v = getattr(b, k)
        setattr(rows, k, v[:, :3 * n] if k in ("out", "xb") else v[:3 * n])
    ratios = _ratios(pipe._iplan, rows, ref)
    record_property("ratio", f"{max(ratios.values()):.4f}")
    _assert_within(ratios, layout)


def _positions(n, seed):
    """Real Hanabi-Full positions: reset + 10 random legal moves; -> (global observation float [n, 785], legal float)."""
    from hanabizero_b200.hanabi_env import HanabiVecEnv
    env = HanabiVecEnv(n, "Hanabi-Full", np.arange(n) + seed)
    g, _, legal = env.reset_all()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(10):
        g, _, legal, _, _, _ = env.step_all(torch.multinomial(legal, 1, generator=gen).view(-1).int(), auto_reset=True)
    env.check()
    return g.clone(), legal.clone()


def test_root_actions_agree_with_the_module_path_at_4096_roots(record_property):
    """4096 Hanabi-Full roots (8 tickets of 512, 50 simulations, fp16 plans, the row-block executor): the arg-max root
    action of submit_observations agrees with the nn.Module path (initial_inference_device + run_multi without plans)
    on at least 99 % of the roots."""
    from hanabizero_b200 import cytree
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    n, G, S, A = 512, 8, 4, 20
    g, legal = _positions(n * G, seed=11)
    frames = g.repeat(1, S)
    model = _model(True, 785, S, A)
    cfg = _cfg("torch_amp", sims=50)
    noise = torch.from_numpy(np.random.default_rng(7).dirichlet([0.3] * A, n * G).astype(np.float32)).cuda()
    pipe = SearchPipeline(MCTS(cfg), model, n, A, depth=2, wave=G, stack=S)
    visits = torch.empty(n * G, A, dtype=torch.int32, device="cuda")
    for k in range(G):
        rows = slice(k * n, (k + 1) * n)
        pipe.submit_observations(0.25, noise[rows], frames[rows], legal[rows], visits[rows])
    pipe.drain()
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        _, logits, hidden = model.initial_inference_device(frames)
    roots = cytree.Roots(n * G, A, 50)
    roots.prepare(0.25, noise, torch.zeros(n * G, device="cuda"), logits.float().contiguous(), legal.int())
    MCTS(cfg, use_plan=False).run_multi(roots, model, hidden, use_graph=False)
    vm, _ = roots.get_stats_tensors()
    agree = float((vm.argmax(1) == visits.argmax(1)).float().mean())
    record_property("agreement", f"{agree:.4f}")
    assert agree >= 0.99, agree


def _hidden_ticket(n, A, seed, half):
    g = torch.Generator(device="cuda").manual_seed(seed)
    legal = _legal(n, A, seed)
    hidden = torch.randn(n, 512, device="cuda", generator=g).clamp_min(0) * 0.7
    return dict(noise=torch.rand(n, A, device="cuda"), reward=torch.randn(n, device="cuda", generator=g) * 0.1,
                logits=torch.randn(n, A, device="cuda", generator=g), legal=legal,
                hidden=hidden.half() if half else hidden,
                visits=torch.full((n, A), -1, dtype=torch.int32, device="cuda"),
                values=torch.full((n,), float("nan"), device="cuda"))


def test_hidden_and_observation_tickets_in_one_pipeline():
    """Two hidden-state tickets, two observation tickets, two hidden-state tickets: each change of kind launches the
    open wave (waves of two tickets on slots 0, 1, 0), and every ticket equals its stand-alone equivalent — a hidden-state
    ticket its own Roots(n) + run_multi (row-block executor), an observation ticket the same tickets submitted to a fresh
    pipeline."""
    from hanabizero_b200 import cytree
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    full, D, _, A, _, _, _ = _layout("full-global")
    S, n, G = 4, 128, 4
    model = _model(full, D, S, A)
    make = lambda: SearchPipeline(MCTS(_cfg("torch_amp")), model, n, A, depth=2, executor="rows", wave=G, stack=S)
    pipe = make()
    hid = [_hidden_ticket(n, A, 60 + k, half=k % 2 == 1) for k in range(4)]
    obs = [_obs_ticket(n, S, D, A, 70 + k) for k in range(2)]
    sub_h = lambda t: pipe.submit(0.25, t["noise"], t["reward"], t["logits"], t["legal"], t["hidden"], t["visits"],
                                  t["values"])
    ids = [sub_h(hid[0]), sub_h(hid[1])]
    assert pipe._waves.open["count"] == 2 and pipe._open_kind() == "hidden"
    ids.append(_submit_obs(pipe, obs[0]))
    assert pipe._open_kind() == "obs" and pipe._waves.open["count"] == 1     # the hidden wave launched
    ids.append(_submit_obs(pipe, obs[1]))
    ids += [sub_h(hid[2])]
    assert pipe._open_kind() == "hidden" and pipe._waves.open["count"] == 1
    ids += [sub_h(hid[3])]
    pipe.drain()
    torch.cuda.synchronize()
    assert ids == [0, 1, G, G + 1, 0, 1]
    ref = MCTS(_cfg("torch_amp"))
    for k, t in enumerate(hid):
        roots = cytree.Roots(n, A, SIMS)
        roots.prepare(0.25, t["noise"], t["reward"], t["logits"], t["legal"])
        ref.run_multi(roots, model, t["hidden"], executor="rows")
        v, val = roots.get_stats_tensors()
        assert torch.equal(t["visits"], v) and torch.equal(t["values"].view(torch.int32), val.view(torch.int32)), k
    fresh = make()
    again = [dict(t, visits=torch.empty_like(t["visits"]), values=torch.empty_like(t["values"])) for t in obs]
    for t in again:
        _submit_obs(fresh, t)
    fresh.drain()
    torch.cuda.synchronize()
    for t, u in zip(obs, again):
        assert torch.equal(t["visits"], u["visits"]) and torch.equal(t["values"].view(torch.int32),
                                                                     u["values"].view(torch.int32))


@pytest.mark.parametrize("how", ["sgd step", "load_state_dict"])
def test_weight_updates_after_drain_reach_the_next_observation_wave(how):
    """Update the module after drain(): the next observation wave of the same pipeline equals a freshly built pipeline
    on the updated module, and differs from the wave before the update."""
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    full, D, _, A, _, _, _ = _layout("small-global")
    S, n, G = 2, 128, 2
    model = _model(full, D, S, A, seed=1)
    make = lambda: SearchPipeline(MCTS(_cfg("torch_amp")), model, n, A, depth=2, wave=G, stack=S)
    pipe = make()
    tickets = [_obs_ticket(n, S, D, A, 90 + k) for k in range(G)]
    outputs = lambda: [dict(t, visits=torch.empty_like(t["visits"]), values=torch.empty_like(t["values"])) for t in tickets]
    before = outputs()
    for t in before:
        _submit_obs(pipe, t)
    pipe.drain()
    if how == "sgd step":
        model.train()
        opt = torch.optim.SGD(model.parameters(), lr=0.5)
        x = tickets[0]["frames"].view(n, -1).float()
        state = model.representation(x)
        policy, value = model.prediction(state)
        (policy.square().mean() + value.square().mean() - state.mean()).backward()
        opt.step()
        model.eval()
    else:
        other = _model(full, D, S, A, seed=2)
        model.load_state_dict(other.state_dict())
    after = outputs()
    for t in after:
        _submit_obs(pipe, t)
    pipe.drain()
    fresh_out = outputs()
    fresh = make()
    for t in fresh_out:
        _submit_obs(fresh, t)
    fresh.drain()
    torch.cuda.synchronize()
    for a, f in zip(after, fresh_out):
        assert torch.equal(a["visits"], f["visits"]) and torch.equal(a["values"].view(torch.int32),
                                                                     f["values"].view(torch.int32))
    assert any(not torch.equal(a["values"], b["values"]) for a, b in zip(after, before)), "the update changed nothing"


def _actor_loop(decode, moves=30, games=256, groups=2, S=4):
    """Closed host-driven loop: EnvPipeline(fmt="bits") groups -> host frame stack -> submit_observations -> host arg-max
    -> step.  decode=False hands in the packed rows and the meta rows' legal mask word; decode=True the float frames
    and legal mask unpack_bits decodes from the same rows.  -> (per move: actions, visits), final env dumps."""
    from hanabizero_b200.hanabi_env import EnvPipeline, HanabiVecEnv
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    envs = [HanabiVecEnv(games, "Hanabi-Full", np.arange(games) + 1000 * g) for g in range(groups)]
    for e in envs:
        e.reset_all(observe=False)
    A, D, W = envs[0].num_actions, envs[0].global_dim, envs[0].bits_words - 4
    model = _model(True, D, S, A)
    pipe = SearchPipeline(MCTS(_cfg("torch_amp")), model, games, A, depth=groups, stack=S)
    ep = EnvPipeline(envs, fmt="bits")
    shape = (games, S, D) if decode else (games, S, W)
    stacks = [torch.zeros(shape, dtype=torch.float32 if decode else torch.int32).pin_memory() for _ in range(groups)]
    legal_f = [torch.zeros(games, A).pin_memory() for _ in range(groups)]
    visits = [torch.zeros(games, A, dtype=torch.int32).pin_memory() for _ in range(groups)]
    for g in range(groups):
        ep.observe_now(g)
    log = []
    for move in range(moves):
        for g in range(groups):
            words, meta = ep.wait(g)
            new = meta[:, 2] != 0 if move else torch.ones(games, dtype=torch.bool)
            if decode:
                u = envs[g].unpack_bits(words, meta)
                frame = torch.from_numpy(u["global_obs"]).float()
                legal_f[g].copy_(torch.from_numpy(u["legal"]).float())
            else:
                frame = words
            st = stacks[g]
            st[:, :-1] = st[:, 1:].clone()
            st[:, -1] = frame
            st[new] = frame[new].unsqueeze(1).expand(-1, S, -1)      # a new episode: its first frame fills the stack
            tid = pipe.submit_observations(0.0, None, st, legal_f[g] if decode else meta[:, 0], visits[g])
            pipe.wait(tid)
            acts = visits[g].argmax(1).int()
            log.append((acts.clone(), visits[g].clone()))
            ep.step(g, acts)
    ep.drain()
    for e in envs:
        e.check()
    return log, [e.dump().cpu() for e in envs]


def test_host_driven_actor_loop_bits_and_decoded_floats_agree():
    log_bits, dump_bits = _actor_loop(decode=False)
    log_f32, dump_f32 = _actor_loop(decode=True)
    assert len(log_bits) == len(log_f32) == 60
    for m, ((a0, v0), (a1, v1)) in enumerate(zip(log_bits, log_f32)):
        assert torch.equal(a0, a1) and torch.equal(v0, v1), m
        assert int(v0.sum()) == v0.shape[0] * (SIMS - 1)
    for d0, d1 in zip(dump_bits, dump_f32):
        assert torch.equal(d0, d1)
