"""GPU: root inference as self-play runs it — the byte frame ring gathered into the network input (hz_ring_gather,
hanabizero_b200/csrc/hz_selfplay.cu) and the folded initial plan (InitialPlan, hanabizero_b200/plan.py: BatchNorm folded
into the weights, 10 / 5 cuBLASLt GEMMs) — against ONE reference: a float64 copy of the nn.Module
(copy.deepcopy(net).double().eval()) run through representation() and prediction() on the stacked frames.  The reference
is not the folded plan, so a mistake in InitialPlan.refresh (a BN term dropped, a weight put in the wrong slot, a frame's
columns at the wrong offset) shows here.  Also: hz_ring_gather / hz_ring_refill against torch indexing bit for bit,
SelfPlayEngine's root inference move by move, weight refresh, and the release of the plans' GEMM handles.

Every activation the plan keeps in a buffer is checked, not only the outputs: r1, t1, r2, r3, t2 of the representation,
the state, the heads' hidden layers and the value / policy logits.  A tensor's depth L is the number of GEMMs on its
longest path from the frames: Hanabi-Full r1 1 ... state 6, value logits 9, policy logits 10; Hanabi-Small r1 1, t1 2,
state 3, logits 5.  An error in an early layer is largest right after it and is diluted by the layers behind it: a
dropped BN scale on the first residual block's second layer of Hanabi-Full moves its output r2 by some 20-30 bounds but the
state by only ~6, so checking outputs alone would leave that mistake near the bound.

Tolerances, from the arithmetic.  u is the unit roundoff of the plan's type.
  * fp16 plan (u = 2^-11): every layer rounds its output to fp16 (<= u of the value) and multiplies by folded weights
    rounded to fp16 (<= u per product; their signs are random, so the sum is off by ~u of the output, not by u of
    sum |w x|).  The frames are 0/1, exact in fp16.  cuBLASLt accumulates in fp32 (CUBLAS_COMPUTE_32F): 2^-24 per
    addition over K0 <= 3200 terms is negligible next to u.  Eval-mode BN keeps each layer's gain O(1), so the layers'
    errors add rather than multiply: a tensor L layers deep is within ~2 L u of its largest magnitude.  Asserted:
    4 L u max|reference|.
  * fp32 plan (u = 2^-24, CUBLAS_COMPUTE_32F: fp32 products and sums, no TF32): weight and output rounding are u as
    above, but now the accumulation's own rounding is of the same order per addition and no longer negligible.  The
    rounding errors of a K-term sum add up like a random walk, ~sqrt(K) u of its partial sums, and no faster in a
    blocked or split-K order; with K0 <= 3200 (Hanabi-Full local, 4 frames of 800) that is sqrt(3200) = 57 < 64.
    Asserted: 4 L u max|reference| x 64 (headroom 64).
  * Decoded value (hz_support_decode on the plan's own logits): against the float64 decode of those same logits,
    within the decode's own bar (tests/test_nn_glue_gpu.py: 1e-5 relative, 2e-5 absolute per 100 of the support's
    half-width).  The logit bound above already covers the distance to the module.
Negative controls (a frame's weight columns swapped, a BN shift dropped, a BN scale dropped) must exceed their bound by
at least 10x: they guard the bounds against being loosened.  Each check records its largest error / bound ratio as the
test property `ratio` (pytest --junitxml shows it).
"""
import copy
import gc

import numpy as np
import pytest
import torch

from test_nn_glue_gpu import _ref_decode

pytestmark = pytest.mark.gpu

U = {torch.float16: 2.0 ** -11, torch.float32: 2.0 ** -24}
HEADROOM = {torch.float16: 1, torch.float32: 64}
DEPTH = {True: dict(r1=1, t1=2, r2=3, r3=4, t2=5, state=6, actor1=7, value1=7, a1=8, value2=8, a2=9, value=9, policy=10),
         False: dict(r1=1, t1=2, state=3, value1=4, actor1=4, value=5, policy=5)}
SENTINEL = -5.0          # never an activation: every buffer but the logits is >= 0 after its ReLU
# name -> (Hanabi-Full?, frame_dim, frame_stride, actions, support)
LAYOUTS = {"full-global": (True, 785, 800, 20, 201), "full-local": (True, 660, 672, 20, 201),
           "small-global": (False, 193, 208, 11, 51), "small-local": (False, 173, 176, 11, 51)}
DTYPES = {"fp16": torch.float16, "fp32": torch.float32}


def _net(full, inputs, A, support, seed):
    """Random BN statistics and affine terms, output heads re-drawn (the reference zero-initialises them)."""
    from hanabizero_b200.model import MuZeroNet, MuZeroNetFull
    torch.manual_seed(seed)
    net = (MuZeroNetFull if full else MuZeroNet)(inputs, A, support, support)
    net = net.randomize_heads(std=0.05, seed=seed).to("cuda")
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.normal_(0, 0.2); m.running_var.uniform_(0.5, 1.5)
            m.weight.data.uniform_(0.5, 1.5); m.bias.data.normal_(0, 0.2)
    return net.eval()


def _float64(net):
    """The reference module.  Copied before the module's cached plans exist (they own library handles)."""
    assert "_iplans" not in net.__dict__ and "_plans" not in net.__dict__
    return copy.deepcopy(net).double().eval()


@torch.no_grad()
def _reference(net64, frames):
    """float64 module on frames [n, S * D] (oldest first): representation() then prediction(), and every intermediate
    activation the plan keeps, computed with the module's own sub-modules."""
    x = frames.double()
    rep, v, p = net64._representation, net64._prediction_value, net64._prediction_actor
    state = net64.representation(x)
    policy, value = net64.prediction(state)
    act = dict(state=state, value=value, policy=policy)
    r1 = act["r1"] = rep[2](rep[1](rep[0](x)))
    if net64.full:                       # _ResBlock(skip_after_first=False): t = relu(bn1 fc1 x), relu(bn2 fc2 t + x)
        act["t1"] = torch.relu(rep[3].bn1(rep[3].fc1(r1)))
        r2 = act["r2"] = rep[3](r1)
        r3 = act["r3"] = rep[6](rep[5](rep[4](r2)))
        act["t2"] = torch.relu(rep[7].bn1(rep[7].fc1(r3)))
        a1 = act["actor1"] = p[2](p[1](p[0](state)))
        v1 = act["value1"] = v[2](v[1](v[0](state)))
        act["a1"] = torch.relu(p[3].bn1(p[3].fc1(a1)))
        act["a2"] = p[3](a1)
        act["value2"] = v[5](v[4](v[3](v1)))
    else:                                # _ResBlock(skip_after_first=True): t = relu(bn1 fc1 x + x), relu(bn2 fc2 t)
        act["t1"] = torch.relu(rep[3].bn1(rep[3].fc1(r1)) + r1)
        act["value1"] = v[2](v[1](v[0](state)))
        act["actor1"] = p[2](p[1](p[0](state)))
    return act


def _plan_tensors(plan, b):
    """The plan's buffers under the reference's names (head order: Hanabi-Full [actor | value], Hanabi-Small
    [value | actor])."""
    H, W, A = plan.H, plan.n_support, plan.A
    t = dict(r1=b.r1, t1=b.t1, state=b.state, value=b.out[0, :, :W], policy=b.out[1, :, :A])
    if plan.full:
        t.update(r2=b.r2, r3=b.r3, t2=b.t2, actor1=b.h1[:, :H], value1=b.h1[:, H:], a1=b.xb[0], value2=b.xb[1],
                 a2=b.xb[2])
    else:
        t.update(value1=b.h1[:, :H], actor1=b.h1[:, H:])
    return t


def _ratios(plan, b, ref):
    """error / bound of every checked tensor (NaN if the plan produced one: it fails every comparison)."""
    got, out = _plan_tensors(plan, b), {}
    for k, depth in DEPTH[plan.full].items():
        scale = max(ref[k].abs().max().item(), 1e-3)
        bound = 4 * depth * U[plan.dtype] * HEADROOM[plan.dtype] * scale
        out[k] = (got[k].double() - ref[k]).abs().max().item() / bound
    return out


def _worst(ratios):
    k = max(ratios, key=lambda k: ratios[k] if ratios[k] == ratios[k] else float("inf"))
    return k, ratios[k]


def _assert_within(ratios, where):
    bad = {k: round(r, 3) for k, r in ratios.items() if not r <= 1.0}
    assert not bad, f"{where}: error / bound above 1: {bad}"


def _padding_is_zero(plan, b, where):
    W, A = plan.n_support, plan.A
    assert torch.count_nonzero(b.out[0, :, W:]) == 0, f"{where}: value logit padding columns {W}..{plan.P3}"
    assert torch.count_nonzero(b.out[1, :, A:]) == 0, f"{where}: policy logit padding columns {A}..{plan.P3}"


def _frames(n, S, D, seed):
    """0/1 frames [n, S, D] (density 0.2); column j of frame j is 1 and columns 0..S-1 are otherwise 0, so the frames
    of a row all differ."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    f = (torch.rand(n, S, D, device="cuda", generator=g) < 0.2).to(torch.uint8)
    f[:, :, :S] = torch.eye(S, dtype=torch.uint8, device="cuda")
    return f


def _ring(frames, stride, head):
    """uint8 ring [n, S, stride]: logical frame j in slot (head + j) % S, padding bytes 0."""
    n, S, D = frames.shape
    ring = torch.zeros(n, S, stride, dtype=torch.uint8, device="cuda")
    for j in range(S):
        ring[:, (head + j) % S, :D] = frames[:, j]
    return ring


def _gather(ring, head, out, ld_out, frame_stride, n=None):
    from hanabizero_b200 import _lib
    n = ring.shape[0] if n is None else n
    _lib.check(_lib.load().hz_ring_gather(torch.cuda.current_stream().cuda_stream, ring.data_ptr(), head, out.data_ptr(),
                                          ld_out, frame_stride, n, ring.shape[1], ring.shape[2], out.element_size()))


def _run(plan, ring, head):
    """Gather the ring into bound(n).x and run the plan on it, every buffer pre-filled with a sentinel.  -> (bound,
    decoded value)."""
    n = ring.shape[0]
    b = plan.bound(n)
    for t in (b.x, b.state, b.h1, b.out, b.r1, b.t1) + ((b.r2, b.r3, b.t2, b.xb) if plan.full else ()):
        t.fill_(SENTINEL)
    _gather(ring, head, b.x, b.x.stride(0), plan.frame_stride)
    value, _, _ = plan.run(n, decode_value=True)
    torch.cuda.synchronize()
    return b, value


def _check_value(plan, b, value):
    half = plan.support.abs().max().item()
    want = _ref_decode(b.out[0, :, :plan.n_support], plan.support, plan.net.support_delta)
    torch.testing.assert_close(value.double(), want, rtol=1e-5, atol=2e-5 * max(1.0, half / 100))


def _check(plan, b, value, ref, where, record=None):
    ratios = _ratios(plan, b, ref)
    if record is not None:
        k, r = _worst(ratios)
        record("ratio", f"{r:.4f} ({k})")
    _assert_within(ratios, where)
    _padding_is_zero(plan, b, where)
    if value is not None:
        _check_value(plan, b, value)
    return ratios


def _case(layout, S, dtype, n, seed, A=None, support=None, record=None):
    from hanabizero_b200.plan import InitialPlan
    full, D, stride, A0, sup0 = LAYOUTS[layout]
    A, support = A or A0, support or sup0
    net = _net(full, D * S, A, support, seed)
    net64 = _float64(net)
    plan = InitialPlan(net, dtype, D, S)
    assert (plan.frame_stride, plan.K0) == (stride, S * stride)
    frames = _frames(n, S, D, seed)
    head = S - 1                                   # logical frame j in slot (S - 1 + j) % S: the gather wraps
    b, value = _run(plan, _ring(frames, stride, head), head)
    want_x = torch.zeros(n, S, stride, dtype=dtype, device="cuda")
    want_x[:, :, :D] = frames
    assert torch.equal(b.x.view(n, S, stride), want_x), "gathered input"
    ref = _reference(net64, frames.view(n, -1))
    _check(plan, b, value, ref, f"{layout} S={S} {dtype} n={n}", record)
    return net, plan, b, frames, ref


# ---- every frame layout x stack x type ----------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("S", [1, 3, 4])
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_initial_plan_matches_float64_module_at_every_layout(layout, S, dtype, record_property):
    """Global and local (POMDP) frames of both networks, 1, 3 and 4 frames (K0 from 176 to 3200), 300 rows."""
    _case(layout, S, DTYPES[dtype], 300, seed=S * 10 + len(layout), record=record_property)


# (layout, A, support, P3): P3 = round_up(max(support, A), 16); (11, 9) has more policy logits than support bins
WIDTHS = [("full-global", 20, 201, 208), ("full-global", 32, 21, 32), ("small-global", 11, 51, 64),
          ("small-global", 11, 9, 16)]


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("layout,A,support,p3", WIDTHS)
def test_initial_plan_output_widths(layout, A, support, p3, dtype, record_property):
    _, plan, _, _, _ = _case(layout, 4, DTYPES[dtype], 300, seed=A + support, A=A, support=support,
                             record=record_property)
    assert (plan.A, plan.n_support, plan.P3) == (A, support, p3)


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("n", [1, 5, 77, 1000, 4096 + 77])
@pytest.mark.parametrize("layout", ["full-local", "small-global"])
def test_initial_plan_across_row_counts(layout, n, dtype, record_property):
    """cuBLASLt picks its kernels by row count: one row, a few, and batches past 4096."""
    _case(layout, 4, DTYPES[dtype], n, seed=n, record=record_property)


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_ring_padding_never_reaches_the_network(layout, dtype):
    """1s written into every padding byte of the ring (columns frame_dim..stride of every slot) reach the gathered
    input but meet zero weight columns: every buffer of the plan is bit-identical to the run with zero padding."""
    _, D, stride, _, _ = LAYOUTS[layout]
    S, head = 4, 3
    net, plan, b, frames, _ = _case(layout, S, DTYPES[dtype], 300, seed=5)
    clean = {k: v.clone() for k, v in _plan_tensors(plan, b).items()}
    ring = _ring(frames, stride, head)
    ring[:, :, D:] = 1
    b2, _ = _run(plan, ring, head)
    assert b2 is b
    assert (b.x.view(-1, S, stride)[:, :, D:] == 1).all(), "the padding bytes must reach the gathered input"
    for k, v in _plan_tensors(plan, b).items():
        assert torch.equal(v, clean[k]), f"{k} changed with 1s in the padding bytes"


# ---- negative controls ----------------------------------------------------------------------------------------------

@torch.no_grad()
def _corrupt(plan, control):
    rep, w, fs, S = plan.net._representation, plan._w, plan.frame_stride, plan.stack
    if control == "frames 0 and S-1 swapped in W0":
        first = w["W0"][:, :fs].clone()
        w["W0"][:, :fs] = w["W0"][:, (S - 1) * fs:]
        w["W0"][:, (S - 1) * fs:] = first
    elif control == "b0 without the BN shift":
        w["b0"].copy_(rep[0].bias)
    elif control == "Wr0b without the BN scale":
        w["Wr0b"].copy_(rep[3].fc2.weight)


CONTROLS = ["frames 0 and S-1 swapped in W0", "b0 without the BN shift", "Wr0b without the BN scale"]


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("layout", ["full-global", "small-global"])
@pytest.mark.parametrize("control", CONTROLS)
def test_negative_controls_fail_the_checker_by_10x(control, layout, dtype, record_property):
    """Corrupt the plan's folded weights in place (refresh() does not see it: the module is unchanged); the checker
    must then report an error of at least 10 bounds."""
    net, plan, b, frames, ref = _case(layout, 4, DTYPES[dtype], 300, seed=9)
    _corrupt(plan, control)
    b2, _ = _run(plan, _ring(frames, plan.frame_stride, 3), 3)
    assert b2 is b and not plan.refresh()
    k, r = _worst(_ratios(plan, b, ref))
    record_property("ratio", f"{r:.4f} ({k})")
    assert r >= 10, f"{control}: largest error / bound {r:.3g} ({k}) is under 10"


# ---- weight refresh -------------------------------------------------------------------------------------------------

def _update(net, how, frames):
    if how == "sgd step":
        net.train()
        opt = torch.optim.SGD(net.parameters(), lr=0.2)
        state = net.representation(frames.float())
        policy, value = net.prediction(state)
        (policy.square().mean(0).sum() + value.square().mean(0).sum() - state.mean(0).sum()).backward()
        opt.step()
        net.eval()
    elif how == "load_state_dict":
        other = _net(net.full, net._representation[0].in_features, net.action_space_n, net._value_support.numel(), 99)
        net.load_state_dict(other.state_dict())
    elif how == "bn running stats":
        with torch.no_grad():
            for m in net.modules():
                if isinstance(m, torch.nn.BatchNorm1d):
                    m.running_mean.add_(0.3)
                    m.running_var.mul_(1.5)


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("layout", ["full-global", "small-global"])
@pytest.mark.parametrize("how", ["sgd step", "load_state_dict", "bn running stats"])
def test_refresh_follows_in_place_updates(how, layout, dtype, record_property):
    """After an in-place update of the module, refresh() re-folds into the same buffers (the bound's x / state / out
    and every weight tensor keep their addresses, so chains built over them stay valid) and the next run matches the
    updated float64 module — and no longer the old one.  A second refresh() has nothing to do."""
    net, plan, b, frames, old_ref = _case(layout, 4, DTYPES[dtype], 300, seed=13)
    ptrs = {k: v.data_ptr() for k, v in plan._w.items()}
    bptrs = (b.x.data_ptr(), b.state.data_ptr(), b.out.data_ptr())
    flat = frames.view(frames.shape[0], -1)
    _update(net, how, flat)
    assert plan.refresh() is True
    assert plan.refresh() is False
    assert {k: v.data_ptr() for k, v in plan._w.items()} == ptrs
    b2, value = _run(plan, _ring(frames, plan.frame_stride, 3), 3)
    assert b2 is b and (b.x.data_ptr(), b.state.data_ptr(), b.out.data_ptr()) == bptrs
    _check(plan, b, value, _reference(_float64(net), flat), f"after {how}", record_property)
    k, r = _worst(_ratios(plan, b, old_ref))
    assert r > 10, f"{how}: the update moved the outputs by only {r:.3g} bounds ({k}); it tests nothing"


# ---- hz_ring_gather / hz_ring_refill, bit for bit --------------------------------------------------------------------

DP = 208


@pytest.mark.parametrize("elem_bytes", [2, 4])
@pytest.mark.parametrize("S", [1, 3, 4])
def test_ring_gather_equals_torch_indexing(S, elem_bytes):
    """Random bytes (0..255, exact in both output types), every head, 1 / 3 / 5 / 4097 games (4 per CTA: partial
    CTAs), and both the dense layout (frame_stride = padded_dim, ld_out = S * frame_stride) and a spread one whose gap
    columns (between frames and after the last) must keep their sentinel.  One game more is allocated than gathered:
    its output row must stay untouched."""
    dtype = torch.float16 if elem_bytes == 2 else torch.float32
    g = torch.Generator(device="cuda").manual_seed(S * 10 + elem_bytes)
    for n in (1, 3, 5, 4097):
        ring = torch.randint(0, 256, (n + 1, S, DP), dtype=torch.uint8, device="cuda", generator=g)
        for head in range(S):
            for fs, ld in ((DP, S * DP), (DP + 32, S * (DP + 32) + 48)):
                out = torch.full((n + 1, ld), SENTINEL, dtype=dtype, device="cuda")
                _gather(ring, head, out, ld, fs, n=n)
                want = torch.full_like(out, SENTINEL)
                for j in range(S):
                    want[:n, j * fs:j * fs + DP] = ring[:n, (head + j) % S].to(dtype)
                assert torch.equal(out, want), (n, head, fs, ld)


@pytest.mark.parametrize("S", [1, 3, 4])
def test_ring_refill_equals_torch_indexing(S):
    """Every source slot, with done NULL (every game) and with a mask of 0 / 1 / 255 bytes (any non-zero byte means
    done): refilled games hold the source slot's frame in every slot, the others stay byte-identical, and so does the
    game past `num`."""
    from hanabizero_b200 import _lib
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(S)
    for n in (1, 3, 5, 4097):
        base = torch.randint(0, 256, (n + 1, S, DP), dtype=torch.uint8, device="cuda", generator=g)
        mask = torch.tensor([0, 1, 255], dtype=torch.uint8, device="cuda")[
            torch.randint(0, 3, (n,), device="cuda", generator=g)]
        for src in range(S):
            for done in (None, mask):
                ring = base.clone()
                _lib.check(lib.hz_ring_refill(torch.cuda.current_stream().cuda_stream, ring.data_ptr(), src,
                                              None if done is None else done.data_ptr(), n, S, DP))
                want = base.clone()
                sel = torch.zeros(n + 1, dtype=torch.bool, device="cuda")
                sel[:n] = True if done is None else done != 0
                want[sel] = base[sel][:, src:src + 1].expand(-1, S, -1)
                assert torch.equal(ring, want), (n, src, done is None)


# ---- SelfPlayEngine's root inference, move by move ------------------------------------------------------------------

@pytest.mark.parametrize("amp", ["torch_amp", "none"])
@pytest.mark.parametrize("S", [1, 3, 4])
@pytest.mark.parametrize("game,mdp", [("Hanabi-Full", "local"), ("Hanabi-Small", "global")])
def test_selfplay_engine_root_inference_matches_float64_module(game, mdp, S, amp, record_property):
    """The fast path (byte ring + InitialPlan, fp16 plan for amp_type "torch_amp", fp32 for "none") played until a
    game has finished and been re-dealt, one move past that (its stack refilled), and at least 2 S + 1 moves (the ring
    head has gone round twice and every slot holds a frame of its own).  Every move's root inference —
    the bound's buffers after the step — matches the float64 module on the frames the move started from, and the
    ring's padding bytes stay 0 whatever the env kernel writes."""
    from hanabizero_b200.mcts import SearchConfig
    from hanabizero_b200.selfplay import SelfPlayEngine
    full = game == "Hanabi-Full"
    D = {("Hanabi-Full", "local"): 660, ("Hanabi-Small", "global"): 193}[game, mdp]
    A, support, N = (20, 201, 128) if full else (11, 51, 128)
    net = _net(full, D * S, A, support, seed=S)
    net64 = _float64(net)
    eng = SelfPlayEngine(N, game, net, SearchConfig(num_simulations=4, amp_type=amp), seeds=np.arange(N) + 7, mdp=mdp,
                         stack=S)
    assert eng.iplan is not None and eng.iplan.dtype == (torch.float16 if amp == "torch_amp" else torch.float32)
    assert eng.obs_dim == D
    eng.reset()
    finished_at, worst = None, 0.0
    for move in range(60):
        frames = eng.frames_tensor().clone()
        out = eng.step()
        b = eng.iplan.bound(N, owner=eng)
        ratios = _ratios(eng.iplan, b, _reference(net64, frames))
        worst = max(worst, _worst(ratios)[1])
        _assert_within(ratios, f"move {move}")
        _padding_is_zero(eng.iplan, b, f"move {move}")
        assert torch.count_nonzero(eng.ring[:, :, D:]) == 0, f"move {move}: ring padding bytes written"
        if finished_at is not None and move > finished_at and move >= 2 * S:
            break
        if finished_at is None and bool(out["done"].any()):
            finished_at = move
    record_property("ratio", f"{worst:.4f}")
    record_property("moves", move + 1)
    assert finished_at is not None, "no game finished in 60 moves"
    eng.env.check()


# ---- InitialPlan releases its GEMM plans ------------------------------------------------------------------------------

class _CountingLib:
    """plan.lib with hz_gemm_plan_create / hz_gemm_plan_destroy counted."""

    def __init__(self, lib):
        self._lib, self.created, self.destroyed = lib, 0, 0

    def hz_gemm_plan_create(self, *args):
        rc = self._lib.hz_gemm_plan_create(*args)
        self.created += rc == 0
        return rc

    def hz_gemm_plan_destroy(self, h):
        self.destroyed += 1
        return self._lib.hz_gemm_plan_destroy(h)

    def __getattr__(self, name):
        return getattr(self._lib, name)


class _Owner:
    pass


def test_initial_plan_releases_the_gemm_plans_it_drops():
    """Every bound owns a cuBLASLt handle and a 32 MB workspace.  Bounds of owners that have been collected are released
    at the next bound() call (not when the 16-entry cache evicts them); bounds evicted or cleared from the cache are
    released with the object.  In the end every hz_gemm_plan_create has its hz_gemm_plan_destroy."""
    from hanabizero_b200.plan import InitialPlan
    plan = InitialPlan(_net(False, 193, 11, 51, seed=3), torch.float16, 193, 1)
    lib = plan.lib = _CountingLib(plan.lib)
    owners = [_Owner() for _ in range(10)]
    for o in owners:
        plan.bound(64, owner=o)
    plan.bound(64)
    assert (lib.created, lib.destroyed, len(plan._bound)) == (11, 0, 11)
    assert plan.bound(64, owner=owners[3]) is plan._bound[(64, id(owners[3]))]     # live owners keep their entries
    del owners, o
    gc.collect()
    plan.bound(64)                                     # a cache hit still drops the dead owners' entries
    assert (lib.created, lib.destroyed, len(plan._bound)) == (11, 10, 1)
    for i in range(20):                                # short-lived owners: each one's entry goes at the next call
        plan.bound(32 + i, owner=_Owner())
    for n in range(1, 21):                             # 20 distinct n: the cache evicts past 16 entries
        plan.bound(n)
    assert len(plan._bound) == 16
    assert lib.destroyed == lib.created - 16
    plan._bound.clear()
    gc.collect()
    assert lib.created == 11 + 20 + 20 and lib.destroyed == lib.created
