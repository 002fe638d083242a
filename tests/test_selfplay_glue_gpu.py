"""GPU: the three small kernels between a search and the next move or training target, against the exact references of
tests/test_selfplay_glue_reference_cpu.py (whose docstring derives every bound used here).

  * hz_select_action: every A from 1 to 32; temperatures 1, 0.5, 0.25 (the schedule), the non-dyadic 0.1, 0.3, 0.75,
    2.0, a per-row tensor and temperatures so small that c^(1/T) overflows; counts up to 2^20, ties at the maximum,
    counts on illegal moves, rows left without visits; uniforms exactly on every cdf step, one double ulp either side,
    0 and nextafter(1, 0).  Actions and zeroed counts bit for bit, entropy within half a float32 ulp + 2^-42 (1 + H).
    The reference raises each count to 1 / T with the device's own pow (torch.pow on the GPU; checked to be within one
    ulp of Python's), so a cdf step placed exactly on u tests the kernel's sampling, not two libms' last bits.
  * visit_policy_row through hz_visit_policy (float64 and float32), hz_wave_policy and TrajectoryRecorder.flush:
    bit for bit against Fraction(c, s), with counts up to 2^31 - 1 and row sums past 2^32.
  * hz_support_decode: fp16 / fp32, widths 1 ... 256, delta 0.1 ... 3 on the model's support, against decode_ref within
    its bound; the largest error / bound ratio of each case is printed and recorded as the test property `ratio`.  And
    the fused search step at delta 0.1 on the same row regimes, bit for bit against hz_support_decode's values.
"""
import math

import numpy as np
import pytest
import torch

from test_selfplay_glue_reference_cpu import (decode_ref, entropy_bound, policy_ref, select_action_defined,
                                              step_uniforms)

pytestmark = pytest.mark.gpu

TEMPS = [1.0, 0.5, 0.25, 0.1, 0.3, 0.75, 2.0]
TINY = [1e-2, 1e-3, 1e-5]


def _count_rows(A, rng):
    """(counts int32 [R, A], legal float32 [R, A]) over the count regimes."""
    rows, legal = [], []

    def add(c, lg=None):
        rows.append(np.asarray(c, np.int64))
        legal.append(np.ones(A, np.float32) if lg is None else np.asarray(lg, np.float32))

    for _ in range(3):
        c = rng.integers(0, 50, A)
        c[rng.random(A) < 0.4] = 0
        c[rng.integers(0, A)] += 1
        add(c)
        add(rng.integers(0, 2 ** 20 + 1, A))                               # sums of c^4 far past 2^53
    add(2 ** 20 - rng.integers(0, 3, A))                                   # near-equal large counts, ties
    c = rng.integers(0, 40, A)
    c[rng.choice(A, min(A, 3), replace=False)] = 40                        # ties at the maximum: the first wins
    add(c)
    add(np.full(A, 8192) if A < 4 else np.r_[[8192, 8192], np.ones(A - 2, np.int64)])   # the order-visible sum
    c = np.zeros(A, np.int64)
    c[rng.integers(0, A)] = 7
    add(c)                                                                 # a single non-zero entry
    c = rng.integers(0, 30, A)
    lg = (rng.random(A) < 0.6).astype(np.float32)
    c[rng.integers(0, A)] = 99                                             # the largest count on an illegal move
    lg[int(np.argmax(c))] = 0.0
    if lg.sum() == 0 and A > 1:
        lg[(int(np.argmax(c)) + 1) % A] = 1.0
    add(c, lg)
    add(rng.integers(1, 9, A), np.zeros(A))                                # every visit illegal: no move
    add(np.zeros(A, np.int64))                                             # no visits at all
    return np.stack(rows).astype(np.int32), np.stack(legal)


class _DevicePow:
    """c ** e as the device computes it (torch.pow on float64 CUDA tensors), checked against Python's pow.  At e = 1
    the kernel takes c itself, as Python's c ** 1.0 does (torch.pow(c, 1.0) is not always exactly c)."""

    def __init__(self, counts, exponents):
        self.table = {}
        for e in sorted(set(exponents) - {1.0}):
            cs = sorted(set(int(c) for c in np.asarray(counts).ravel()))
            t = torch.tensor(cs, dtype=torch.float64, device="cuda")
            got = torch.pow(t, torch.full_like(t, e)).cpu().tolist()
            for c, g in zip(cs, got):
                try:
                    h = float(c) ** e
                except OverflowError:
                    h = math.inf
                assert g == h or abs(g - h) <= math.ulp(h), (c, e, g, h)       # a faithful pow on both sides
                self.table[(c, e)] = g

    def __call__(self, c, e):
        return float(c) if e == 1.0 else self.table[(int(c), e)]


def _select(visits, legal, temperature, uniforms):
    from hanabizero_b200.selfplay import select_action_batch
    v = torch.from_numpy(visits).cuda()
    act, ent = select_action_batch(v, torch.from_numpy(legal).cuda(), temperature, uniforms is None, uniforms)
    return act.cpu().numpy(), ent.cpu().numpy(), v.cpu().numpy()


def _check_rows(visits, legal, temps, uniforms, act, ent, v_after, power):
    for i in range(visits.shape[0]):
        u = None if uniforms is None else float(uniforms[i])
        a, h, c = select_action_defined(visits[i].tolist(), legal[i].tolist(), temps[i], u, power)
        assert act[i] == a, (i, temps[i], u, visits[i].tolist(), legal[i].tolist(), act[i], a)
        assert v_after[i].tolist() == c, i
        if a < 0:
            assert math.isnan(ent[i]), (i, ent[i])
        else:
            assert abs(float(ent[i]) - h) <= entropy_bound(h), (i, float(ent[i]), h, entropy_bound(h))


@pytest.mark.parametrize("A", range(1, 33))
def test_select_action_deterministic(A):
    rng = np.random.default_rng(1000 + A)
    visits, legal = _count_rows(A, rng)
    R = visits.shape[0]
    per_row = rng.choice(TEMPS + TINY, R)
    power = _DevicePow(visits, [1 / t for t in TEMPS + TINY])
    for T in TEMPS + TINY + ["rows"]:
        temps = per_row if T == "rows" else np.full(R, T)
        arg = torch.from_numpy(per_row) if T == "rows" else T
        act, ent, v_after = _select(visits.copy(), legal, arg, None)
        _check_rows(visits, legal, temps, None, act, ent, v_after, power)
    assert (act[-2:] == -1).all()


@pytest.mark.parametrize("A", range(1, 33))
def test_select_action_samples_on_the_cdf_steps(A):
    rng = np.random.default_rng(2000 + A)
    visits, legal = _count_rows(A, rng)
    power = _DevicePow(visits, [1 / t for t in TEMPS + TINY])
    for T in TEMPS + TINY + ["rows"]:
        rv, rl, rt, ru = [], [], [], []
        for i in range(visits.shape[0]):
            t = float(rng.choice(TEMPS)) if T == "rows" else T
            a, _, _ = select_action_defined(visits[i].tolist(), legal[i].tolist(), t, None, power)
            if a < 0:
                us = [0.0, 0.5]
            else:
                probs = _probs(visits[i], legal[i], t, power)
                us = step_uniforms(probs)
            for u in us:
                rv.append(visits[i]); rl.append(legal[i]); rt.append(t); ru.append(u)
        vv, ll, tt, uu = np.stack(rv), np.stack(rl), np.asarray(rt), np.asarray(ru)
        arg = torch.from_numpy(tt) if T == "rows" else T
        act, ent, v_after = _select(vv.copy(), ll, arg, torch.from_numpy(uu))
        _check_rows(vv, ll, tt, uu, act, ent, v_after, power)


def _probs(counts, legal, t, power):
    from test_selfplay_glue_reference_cpu import ref_select_action
    return ref_select_action(counts.tolist(), legal.tolist(), t, None, power)[1]


def test_undefined_move_stops_the_env():
    """Action -1 from a row without visits is an illegal move: the env's sticky error raises at check()."""
    from hanabizero_b200 import _lib
    from hanabizero_b200.hanabi_env import HanabiVecEnv
    from hanabizero_b200.selfplay import select_action_batch
    N = 4
    env = HanabiVecEnv(N, "Hanabi-Small", np.arange(N), device=torch.device("cuda"))
    _, _, legal = env.reset_all()
    visits = torch.zeros(N, legal.shape[1], dtype=torch.int32, device="cuda")
    visits[:, 0] = 5
    visits[2] = 0
    act, ent = select_action_batch(visits, legal, 1.0, deterministic=True)
    assert act[2].item() == -1 and math.isnan(ent[2].item())
    env.step_all(act, auto_reset=True)
    with pytest.raises(_lib.IllegalMoveError):
        env.check()


# ---- policy targets ---------------------------------------------------------------------------------------------
def _policy_rows(A, rng):
    rows = [rng.integers(0, 2 ** 31, A), np.full(A, 2 ** 31 - 1), rng.integers(0, 300, A), np.zeros(A, np.int64),
            rng.integers(2 ** 30, 2 ** 31, A)]
    one = np.zeros(A, np.int64)
    one[rng.integers(0, A)] = 2 ** 31 - 1
    rows.append(one)
    one = np.zeros(A, np.int64)
    one[-1] = 1
    rows.append(one)
    for _ in range(40):
        rows.append(rng.integers(0, 2 ** 31, A) >> rng.integers(0, 31, A))
    v = np.stack(rows).astype(np.int32)
    mask = (rng.random(len(rows)) < 0.8).astype(np.uint8)
    mask[3] = 1                                                            # the kept zero-sum row
    mask[4] = 0
    return v, mask


def _policy_want(v, mask):
    want64 = np.empty(v.shape, np.float64)
    want32 = np.empty(v.shape, np.float32)
    for i in range(v.shape[0]):
        d, f = policy_ref(v[i].tolist(), bool(mask[i]))
        want64[i], want32[i] = d, f
    return want64, want32


def _same(a, b):
    num = ~np.isnan(b)
    return np.array_equal(a, b, equal_nan=True) and np.array_equal(np.signbit(a[num]), np.signbit(b[num]))


@pytest.mark.parametrize("A", [1, 2, 20, 32])
def test_visit_policy_is_exact(A):
    from hanabizero_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(3000 + A)
    v, mask = _policy_rows(A, rng)
    assert v.astype(np.int64).sum(1).max() > 2 ** 32 or A <= 2
    want64, want32 = _policy_want(v, mask)
    N = v.shape[0]
    dv, dm = torch.from_numpy(v).cuda(), torch.from_numpy(mask).cuda()
    st = torch.cuda.current_stream().cuda_stream
    for m in (dm, None):
        out64 = torch.empty(N, A, dtype=torch.float64, device="cuda")
        out32 = torch.empty(N, A, dtype=torch.float32, device="cuda")
        _lib.check(lib.hz_visit_policy(st, dv.data_ptr(), None if m is None else m.data_ptr(), N, A, out64.data_ptr(),
                                       out32.data_ptr()))
        w64, w32 = (want64, want32) if m is not None else _policy_want(v, np.ones(N, np.uint8))
        assert _same(out64.cpu().numpy(), w64)
        assert _same(out32.cpu().numpy(), w32)
    assert np.isnan(want64[3]).all()


@pytest.mark.parametrize("A", [1, 2, 20, 32])
def test_wave_policy_is_exact(A):
    from hanabizero_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(4000 + A)
    G, count = 3, 2
    v, mask = _policy_rows(A, rng)
    n = v.shape[0]
    stats = torch.from_numpy(np.concatenate([v, v[::-1]] + [np.zeros_like(v)] * (G - 2))).cuda()
    masks = [torch.from_numpy(mask).cuda(), None]
    outs = [torch.full((n, A), -1.0, dtype=torch.float64, device="cuda") for _ in range(count)]
    table = (_lib.PolicyTicket * count)(*[_lib.PolicyTicket(None if m is None else m.data_ptr(), o.data_ptr())
                                          for m, o in zip(masks, outs)])
    _lib.check(lib.hz_wave_policy(torch.cuda.current_stream().cuda_stream, 0, table, count, G, n, A, stats.data_ptr()))
    assert _same(outs[0].cpu().numpy(), _policy_want(v, mask)[0])
    assert _same(outs[1].cpu().numpy(), _policy_want(np.ascontiguousarray(v[::-1]), np.ones(n, np.uint8))[0])


@pytest.mark.parametrize("A", [1, 2, 20, 32])
def test_recorder_flush_targets_are_exact(A):
    from hanabizero_b200.trajectory import TrajectoryRecorder
    rng = np.random.default_rng(5000 + A)
    N, D, T = 3, 16, 5
    rec = TrajectoryRecorder(N, D, A, stack=2, max_len=16, device=torch.device("cuda"))
    cuda = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    rec.begin(cuda(np.zeros((N, D), np.float32)), cuda(np.ones((N, A), np.float32)))
    v, _ = _policy_rows(A, rng)
    v = v[np.r_[0:3, 5:len(v)]][:N * T].reshape(T, N, A)                # the zero-sum row left out (no search gives it)
    for t in range(T):
        rec.append(cuda(np.zeros(N, np.int32)), cuda(np.zeros((N, D), np.float32)), cuda(np.ones((N, A), np.float32)),
                   cuda(np.zeros(N, np.int32)), cuda(v[t]), cuda(np.zeros(N, np.float32)),
                   cuda(np.full(N, t == T - 1, np.uint8)))
    eps = rec.flush()
    assert len(eps) == N
    for ep in eps:
        want = _policy_want(v[:, ep["game"]], np.ones(T, np.uint8))[0]
        assert _same(ep["vis"], want)


# ---- support decode ---------------------------------------------------------------------------------------------
def _support(W, delta):
    """The model's support: arange(-h, h + 1) * delta in float32 (even widths: arange(W) - (W - 1) // 2)."""
    return (torch.arange(W, dtype=torch.float32) - (W - 1) // 2) * delta


def decode_regimes(gen, R, W, dtype):
    """[R, W] float32 logits, a seeded mix of: randn*3; one column above the rest by 5 / 20 / 90 / 110; fp16-range
    magnitudes near +-60000 with small spreads; all equal; one end column dominating (+-h); one-hot on a support point;
    some -inf; one +inf; all -inf."""
    x = torch.randn(R, W, generator=gen) * 3
    kind = torch.randint(0, 12, (R,), generator=gen)
    col = torch.randint(0, W, (R,), generator=gen)
    base = torch.randn(R, W, generator=gen)
    rows = torch.arange(R)
    for k, lift in ((1, 5.0), (2, 20.0), (3, 90.0), (4, 110.0)):
        sel = kind == k
        x[sel] = base[sel]
        x[rows[sel], col[sel]] += lift
    sel = kind == 5
    sign = torch.where(torch.rand(R, generator=gen) < 0.5, -1.0, 1.0)
    spread = torch.randint(0, 4, (R, W), generator=gen).float() * 32.0      # the fp16 grid at 2^15 .. 2^16
    x[sel] = (sign[:, None] * 60000.0 + spread)[sel]
    x[kind == 6] = 1.5
    sel = kind == 7
    x[sel] = base[sel] - 120.0
    x[rows[sel], torch.where(torch.rand(R, generator=gen) < 0.5, 0, W - 1)[sel]] = 0.0
    sel = kind == 8
    x[sel] = -200.0
    x[rows[sel], col[sel]] = 0.0
    some = torch.rand(R, W, generator=gen) < 0.3
    x[(kind == 9)[:, None] & some & (torch.arange(W)[None] != col[:, None])] = -math.inf
    x[rows[kind == 10], col[kind == 10]] = math.inf
    x[kind == 11] = -math.inf
    return x.to(dtype).float()


@pytest.mark.parametrize("delta", [0.1, 0.5, 1.0, 3.0])
@pytest.mark.parametrize("W", [1, 8, 9, 21, 51, 201, 255, 256])
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_support_decode_within_the_derived_bound(dtype, W, delta, record_property):
    from hanabizero_b200 import _lib
    lib = _lib.load()
    gen = torch.Generator().manual_seed(W * 10 + int(delta * 10))
    R = 3000
    x = decode_regimes(gen, R, W, dtype)
    support = _support(W, delta)
    ld = (W + 7) // 8 * 8
    dx = torch.full((R, ld), float("nan"), dtype=dtype, device="cuda")
    dx[:, :W] = x.to(dtype).cuda()
    out = torch.empty(R, device="cuda")
    _lib.check(lib.hz_support_decode(torch.cuda.current_stream().cuda_stream, dx.data_ptr(), dx.element_size(),
                                     support.cuda().data_ptr(), out.data_ptr(), R, W, ld, delta))
    want, bound = decode_ref(x.double().numpy(), support.double().numpy(), delta)
    got = out.double().cpu().numpy()
    err = np.abs(got - want)
    zero = bound == 0                                                        # NaN in the reference: exactly 0
    assert (got[zero] == 0).all()
    ratio = np.where(zero, 0.0, err / np.where(zero, 1.0, bound))
    worst = float(ratio.max())
    record_property("ratio", worst)
    print(f"decode {dtype} W={W} delta={delta}: max error / bound {worst:.3g}")
    assert worst <= 1.0, (int(ratio.argmax()), got[ratio.argmax()], want[ratio.argmax()], bound[ratio.argmax()])


def decode_regime_search_rows(gen, S, N, A, W):
    """Network outputs for the fused step: value / reward rows from decode_regimes, randn policy logits."""
    dev = gen.device
    cpu = torch.Generator().manual_seed(int(torch.randint(0, 2 ** 31, (1,), device=dev, generator=gen).item()))
    v = decode_regimes(cpu, S * N, W, torch.float16).view(S, N, W)
    r = decode_regimes(cpu, S * N, W, torch.float16).view(S, N, W)
    return v.to(dev), r.to(dev), torch.randn(S, N, A, device=dev, generator=gen)


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_fused_step_decodes_at_delta_0_1(dtype):
    """The fused step's values equal hz_support_decode's bit for bit on the decode regimes at the model's delta = 0.1
    support (the lock-step harness feeds the oracle hz_support_decode's values and compares every statistic)."""
    from test_search_step_edges_gpu import lockstep, make_inputs
    lockstep(make_inputs(37, 20, 40, W=201, dtype=dtype, seed=1100, rows=decode_regime_search_rows),
             support_scale=0.1, support_delta=0.1)
