"""CPU: the references that tests/test_selfplay_glue_gpu.py holds the self-play glue kernels to, checked here against
exact arithmetic.  Nothing in this file needs a GPU.

select_action (core/utils.py:280-295; hz_select_action, hanabizero_b200/csrc/hz_selfplay.cu)
  ref_select_action ports it with Python floats: illegal counts zeroed, p[a] = c[a] ** (1 / T) (int ** float: the
  platform's pow, OverflowError when the power is out of range), p[a] / total, first arg-max, and numpy.random.choice's
  own sampling rule for a given uniform u: cdf = cumsum(p); cdf /= cdf[-1]; searchsorted(cdf, u, side='right').
  The sum `total` is taken left to right in ascending action order, as the kernel does and as Python's sum() did up to
  3.11.  Python >= 3.12's built-in sum() of floats is compensated (Neumaier), so it rounds once where the loop rounds
  after every term: the two differ as soon as a partial sum passes 2^53 and drops a term's low bits, e.g. counts
  [8192, 8192, 1, 1] at T = 0.25 give 2^53 for the loop and 2^53 + 2 for sum() (test_sum_order_is_ascending_not_sum).
  Counts below 2^53 ** T never get there.  numpy's cumsum is the same left-to-right loop, so cdf[-1] equals `total`
  recomputed from the p's, which the kernel also recomputes.
  Where the reference raises (ZeroDivisionError for a row without visits, OverflowError when c ** (1 / T)
  overflows) the kernel defines the row as action -1 with NaN entropy; select_action_defined is that contract.  A
  row whose terms are finite but whose sum overflows is undefined there too (the reference's np.random.choice would
  reject its probabilities).

Entropy: entropy_bits = -fsum(p log p) / ln 2 over the float64 p's, so it is the exact entropy of those p's to within
  the rounding of each double log.  The kernel sums -p ln p in double (A <= 32 terms, all >= 0), divides by ln 2 and
  rounds to float32.  Its p's differ from the port's by at most the pow error (2 ulp on the device, 0.52 on the host),
  the sum's A - 1 roundings and one division: 70 * 2^-53 relative.  A relative error r of p moves -p ln p by
  r p |ln p + 1|, so the double entropy is off by at most 2^-45 (H_nats + 1) including the log and the sum, i.e.
  2^-43 (1 + H_bits) after the division by ln 2.  Bound: half a float32 ulp of the result + 2^-42 (1 + H).

Policy targets (visit_policy_row, hz_common.cuh): Fraction(c, s) rounded to double (Python's int / int) and that double
  rounded to float32 (out32 is the float32 of the double target).  A kept row with s = 0 is all NaN.

Support decode (hz_decode.cuh; hz_support_decode and the fused search step): decode_ref evaluates in float64
    E = sum_k softmax(x)_k sp_k,  v = E / delta,  out = sign(v) ((sqrt(1 + 4 eps (|v| + 1 + eps)) - 1) / (2 eps))^2 - 1) delta
  with eps = 0.001, in the cancellation-free form u (u + 2), u = 2 |v| / (s + 1 + 2 eps), checked below against a
  50-digit decimal evaluation of the textbook form.  delta is the float32 the kernel receives; NaN -> 0 as nan_to_num.
  Error bound of the kernel (u32 = 2^-24), with d_k = max(x) - x_k >= 0 and w_k = exp(-d_k):
  * term k is ex2.approx.ftz(fma(x_k, L, -fl(m L))), L = fl32(log2 e).  fl(m L) shifts every exponent by the same
    amount, a common factor that cancels in E.  L differs from log2 e by rho = L ln 2 - 1 = -1.34e-8 relative, the fma
    rounds the exponent (~d_k L) by u32, and ex2.approx is within 2 ulp (2^-22): the term is w_k (1 + eta_k) with
    |eta_k| <= 2^-22 + d_k (|rho| + u32) + 2^-30.
  * ftz: an exponent below -126 (d_k > 87.3) gives 0.  Those terms are below e^-87 of the largest and count as
    eta_k = 1 (entirely lost).
  * sums: a lane adds its 8 terms in order, then 5 butterfly steps: each term sees at most 12 roundings in the sum of
    exponentials and 13 in the fma chain of the weighted sum: gamma_13 = 13 u32 / (1 - 13 u32) of sum w |sp|.
  * E: with Se = sum w, M = sum w |sp| / Se (<= the half-width H), M_eta = sum w |sp| eta / Se and
    eta_e = sum w eta / Se:   |dE| <= M_eta + gamma_13 M + |E| (eta_e + gamma_13 + 2 u32)   (the two divisions).
  * out as a function of E has slope F'(v) = 1 / h'(|out| / delta), h'(x) = 1 / (2 sqrt(|x| + 1)) + eps (<= 1000):
    |d out| <= F'(v) (|dE| (1 + 1e-6) ) + tau |out|.  The float32 transform is cancellation-free, so its own error is
    relative: the additions, square root, division and two products round 9 times, and eps and 1 + 2 eps enter as
    float32 constants (4.7e-8 and u32 relative; out's sensitivity to eps is at most 1): tau = 12 u32 + 5e-8.
  The bound is therefore relative to the output (tau) and to the support's scale through M <= H; the test reports the
  largest error / bound ratio per case.
"""
import math
import sys
from decimal import Decimal, getcontext
from fractions import Fraction

import numpy as np
import pytest

U32 = 2.0 ** -24
EPS = 0.001
RHO = abs(float(np.float32(1.4426950408889634)) * math.log(2) - 1.0)
FTZ_D = 87.0                        # d beyond which a term may be flushed (exponent < -126 at d > 87.3)
G13 = 13 * U32 / (1 - 13 * U32)
TAU = 12 * U32 + 5e-8


# ---- select_action ----------------------------------------------------------------------------------------------
def seq_sum(xs):
    """Left to right, one rounding per term: the kernel's order (and sum() before Python 3.12)."""
    t = 0.0
    for x in xs:
        t += x
    return t


def ref_select_action(counts, legal, temperature, u=None, power=None):
    """core/utils.py:280-295 in Python floats.  u None = deterministic (first arg-max).  Returns
    (action, probabilities, zeroed counts); raises where the reference raises.  power(c, e) replaces `c ** e` (the
    GPU test passes the device's pow, so that a last-bit difference between two libms cannot move a cdf step)."""
    c = [0 if (legal[a] == 0 and int(counts[a]) >= 1) else int(counts[a]) for a in range(len(counts))]
    e = 1 / temperature
    probs = [float(x) ** e if power is None else power(x, e) for x in c]
    total = seq_sum(probs)
    probs = [x / total for x in probs]                      # ZeroDivisionError on a row without visits
    if u is None:
        action = max(range(len(c)), key=lambda a: (c[a], -a))   # np.argmax: the first maximum
    else:
        cdf = []
        run = 0.0
        for p in probs:                                     # np.cumsum
            run += p
            cdf.append(run)
        last = cdf[-1]
        cdf = [x / last for x in cdf]
        action = next((k for k, x in enumerate(cdf) if u < x), len(c))   # searchsorted side='right'
    return action, probs, c


def select_action_defined(counts, legal, temperature, u=None, power=None):
    """The kernel's contract: ref_select_action, or (-1, NaN entropy) where the reference raises or the sum of the
    powers is not finite.  Returns (action, entropy_bits, zeroed counts)."""
    c = [0 if (legal[a] == 0 and int(counts[a]) >= 1) else int(counts[a]) for a in range(len(counts))]
    e = 1 / temperature
    try:
        total = seq_sum(float(x) ** e if power is None else power(x, e) for x in c)
    except OverflowError:
        return -1, math.nan, c
    if not (0 < total < math.inf):
        return -1, math.nan, c
    action, probs, c = ref_select_action(counts, legal, temperature, u, power)
    return action, entropy_bits(probs), c


def entropy_bits(probs):
    return -math.fsum(p * math.log(p) for p in probs if p > 0) / math.log(2)


def entropy_bound(h):
    """|float32 entropy - entropy_bits| (module docstring)."""
    return 0.5 * float(np.spacing(np.float32(h))) + 2.0 ** -42 * (1 + h)


def step_uniforms(probs):
    """Uniforms exactly on every cdf[k] / cdf[-1] (k < A - 1), one double ulp below and above, and 0, nextafter(1, 0)."""
    cdf = np.cumsum(np.asarray(probs, np.float64))
    cdf = cdf / cdf[-1]
    us = {0.0, math.nextafter(1.0, 0.0)}
    for x in cdf[:-1]:
        x = float(x)
        us.update(v for v in (math.nextafter(x, 0.0), x, math.nextafter(x, 1.0)) if 0.0 <= v < 1.0)
    return sorted(us)


# ---- policy targets --------------------------------------------------------------------------------------------
def policy_ref(counts, keep=True):
    """-> (float64 list, float32 array): Fraction(c, s) correctly rounded; zeros when not kept; NaN for s = 0."""
    s = sum(int(c) for c in counts)
    if not keep:
        d = [0.0] * len(counts)
    elif s == 0:
        d = [math.nan] * len(counts)
    else:
        d = [float(Fraction(int(c), s)) for c in counts]
    return d, np.asarray(d, np.float64).astype(np.float32)


# ---- support decode --------------------------------------------------------------------------------------------
def transform64(v, delta):
    """Cancellation-free float64 inverse transform of v (= E / delta), times delta."""
    a = np.abs(v)
    s = np.sqrt(1.0 + 4.0 * EPS * (a + 1.0 + EPS))
    uu = 2.0 * a / (s + (1.0 + 2.0 * EPS))
    r = uu * (uu + 2.0)
    return np.where(v < 0, -r, r) * delta


def decode_ref(x, support, delta):
    """x float64 [R, W] (the logits as the kernel reads them), support float64 [W], delta the float32 the kernel gets.
    -> (out float64 [R], bound float64 [R])."""
    x = np.asarray(x, np.float64)
    sp = np.asarray(support, np.float64)[None, :]
    delta = float(np.float32(delta))
    with np.errstate(all="ignore"):
        m = x.max(1, keepdims=True)
        d = m - x
        w = np.exp(-d)
        se = w.sum(1)
        e = (w * sp).sum(1) / se
        v = e / delta
        out = transform64(v, delta)
        eta = np.where(d > FTZ_D, 1.0, 2.0 ** -22 + d * (RHO + U32) + 2.0 ** -30)
        eta = np.where(np.isnan(eta), 1.0, eta)
        M = (w * np.abs(sp)).sum(1) / se
        M_eta = (w * np.abs(sp) * eta).sum(1) / se
        eta_e = (w * eta).sum(1) / se
        dE = M_eta + G13 * M + np.abs(e) * (eta_e + G13 + 2 * U32)
        slope = 1.0 / (1.0 / (2.0 * np.sqrt(np.abs(out) / delta + 1.0)) + EPS)
        bound = slope * dE * (1 + 1e-6) + TAU * np.abs(out) + 1e-30
    out = np.nan_to_num(out, nan=0.0)
    return out, np.where(np.isnan(bound), 0.0, bound)


def transform_decimal(v):
    """The textbook inverse transform at 50 digits."""
    getcontext().prec = 50
    v = Decimal(v)
    eps = Decimal("0.001")
    r = (((1 + 4 * eps * (abs(v) + 1 + eps)).sqrt() - 1) / (2 * eps)) ** 2 - 1
    return float(-r if v < 0 else r)


def kernel_emulation(x, support, delta, drop_delta=False, s0_one_eps=False):
    """A float32 emulation of the decode's arithmetic (exp correctly rounded; the device's ex2 is within the bound's
    2 ulp), used to show that the bound holds for the kernel's arithmetic and not for its single-line mutations."""
    f = np.float32
    x = np.asarray(x, np.float32)
    sp = np.asarray(support, np.float32)
    L = f(1.4426950408889634)
    outs = []
    for row in x:
        m = row.max()
        nm = f(-m * L)
        arg = (row.astype(np.float64) * float(L) + float(nm)).astype(np.float32)
        ex = np.exp2(arg.astype(np.float64)).astype(np.float32)
        ex[arg < -126] = 0
        se, sw = np.zeros(32, np.float32), np.zeros(32, np.float32)
        for k in range(len(row)):
            lane = k // 8
            se[lane] = f(se[lane] + ex[k])
            sw[lane] = f(float(ex[k]) * float(sp[k]) + float(sw[lane]))
        o = 16
        while o:
            se = (se + se[np.arange(32) ^ o]).astype(np.float32)
            sw = (sw + sw[np.arange(32) ^ o]).astype(np.float32)
            o >>= 1
        eps = f(0.001)
        dl = f(delta)
        v = f(f(sw[0] / se[0]) / dl)
        a = abs(v)
        y = f(f(4 * eps) * f(f(a + f(1)) + eps))
        s = f(np.sqrt(f(f(1) + y)))
        s0 = f(1) + (eps if s0_one_eps else f(f(2) * eps))
        uu = f(f(f(2) * a) / f(s + s0))
        r = f(uu * f(uu + f(2)))
        r = -r if v < 0 else r
        outs.append(float(r if drop_delta else f(r * dl)))
    return np.nan_to_num(np.asarray(outs), nan=0.0)


# ---- tests ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("temperature", [1, 1.0, 0.5, 0.25])
def test_port_matches_exact_rationals_where_the_terms_are_exact(temperature):
    """Integer exponents and sums below 2^53: every power and the total are exact integers, so each probability must
    be the correctly rounded Fraction(c^e, total), the arg-max the first maximum, and the sampled action the first k
    with u < Fraction(cumsum) / Fraction(sum) as numpy rounds them."""
    rng = np.random.default_rng(11)
    e = round(1 / temperature)
    for A in (1, 2, 5, 20, 32):
        for _ in range(60):
            counts = [int(c) for c in rng.integers(0, 3000, A)]
            counts[int(rng.integers(0, A))] += 1
            legal = [1.0] * A
            _, probs, c = ref_select_action(counts, legal, temperature)
            total = sum(x ** e for x in c)
            assert total < 2 ** 53
            assert probs == [float(Fraction(x ** e, total)) for x in c]
            a, _, _ = ref_select_action(counts, legal, temperature)
            assert a == min(k for k in range(A) if c[k] == max(c))
            for u in step_uniforms(probs):
                a, _, _ = ref_select_action(counts, legal, temperature, u)
                cdf = np.cumsum(np.asarray(probs))
                assert a == int(np.searchsorted(cdf / cdf[-1], u, side="right"))


def test_sampling_rule_is_numpy_random_choice():
    """np.random.choice(A, p=p) draws one random_sample() and applies this very rule."""
    rng = np.random.default_rng(12)
    for seed in range(300):
        A = int(rng.integers(1, 33))
        counts = [int(c) for c in rng.integers(0, 60, A)]
        counts[0] += 1
        T = [1.0, 0.5, 0.25, 0.3, 0.75, 2.0][seed % 6]
        _, probs, _ = ref_select_action(counts, [1] * A, T)
        want = np.random.RandomState(seed).choice(A, p=probs)
        u = np.random.RandomState(seed).random_sample()
        assert ref_select_action(counts, [1] * A, T, u)[0] == want


def test_sum_order_is_ascending_not_sum():
    """The kernel's total is the left-to-right sum; Python >= 3.12's sum() is compensated and differs once a partial
    sum passes 2^53."""
    terms = [float(c) ** 4.0 for c in (8192, 8192, 1, 1)]
    assert seq_sum(terms) == 2.0 ** 53
    assert math.fsum(terms) == 2.0 ** 53 + 2
    if sys.version_info >= (3, 12):
        assert sum(terms) == 2.0 ** 53 + 2
    else:
        assert sum(terms) == 2.0 ** 53
    _, probs, _ = ref_select_action([8192, 8192, 1, 1], [1] * 4, 0.25)
    assert probs[2] == 2.0 ** -53


def test_undefined_rows():
    assert select_action_defined([0, 0, 0], [1, 1, 1], 1.0)[:2][0] == -1
    a, h, c = select_action_defined([5, 0, 3], [0, 1, 0], 1.0, 0.5)          # every visit on an illegal move
    assert a == -1 and math.isnan(h) and c == [0, 0, 0]
    with pytest.raises(ZeroDivisionError):
        ref_select_action([5, 0, 3], [0, 1, 0], 1.0)
    with pytest.raises(OverflowError):
        ref_select_action([3, 1000], [1, 1], 0.001)                        # 1000^1000
    assert select_action_defined([3, 1000], [1, 1], 0.001)[0] == -1
    assert select_action_defined([1, 1, 0], [1, 1, 1], 1e-300)[0] == 0     # 1^(1e300) = 1: defined, a tie
    assert select_action_defined([2, 1], [1, 1], 1 / 1023.5)[0] == 0       # 2^1023.5 < DBL_MAX
    assert select_action_defined([2, 1], [1, 1], 1 / 1024.5)[0] == -1      # 2^1024.5 overflows alone
    assert select_action_defined([2, 2], [1, 1], 1 / 1023.5)[0] == -1      # two finite terms, an infinite sum


def test_non_dyadic_temperature_exponent_is_pythons():
    """1 / T in double is what the reference raises counts to; the float32 temperature gives another exponent."""
    for T in (0.1, 0.3):                        # (0.75 and 2.0 are exact in float32)
        assert 1 / T != 1 / float(np.float32(T))
    assert 1 / 0.1 == 10.0 and 1 / float(np.float32(0.1)) < 10.0


def test_entropy_reference_and_bound():
    """entropy_bits equals scipy's base-2 entropy within the bound, and the bound is far below the float32 /ln2 slip."""
    from scipy.stats import entropy
    rng = np.random.default_rng(13)
    for _ in range(500):
        A = int(rng.integers(1, 33))
        counts = [int(c) for c in rng.integers(0, 2 ** 20, A)]
        counts[0] += 1
        _, probs, _ = ref_select_action(counts, [1] * A, [1.0, 0.5, 0.25, 0.1, 0.3][_ % 5])
        h = entropy_bits(probs)
        assert abs(h - entropy(probs, base=2)) <= entropy_bound(h) * 1e-3 + 1e-15
        if h > 1e-6:
            assert abs(h * math.log(2) - h) > 100 * entropy_bound(h)


def test_policy_reference_against_python_division():
    rng = np.random.default_rng(14)
    for A in (1, 2, 20, 32):
        for _ in range(50):
            counts = [int(c) for c in rng.integers(0, 2 ** 31, A)]
            d, f = policy_ref(counts)
            s = sum(counts)
            assert d == [c / s for c in counts]
            assert (f == np.float32(np.asarray(d))).all()
    d, f = policy_ref([0, 0, 0])
    assert all(math.isnan(x) for x in d) and np.isnan(f).all()
    assert policy_ref([3, 4], keep=False)[0] == [0.0, 0.0]


def test_transform_reference_against_decimal():
    vs = [0.0, 1e-9, 1e-4, 0.3, 1.0, 7.5, 100.0, 300.0, 1e4, 3e4] + list(np.random.default_rng(15).normal(0, 50, 200))
    for v in vs:
        for sgn in (1, -1):
            got = float(transform64(np.float64(sgn * v), 1.0))
            want = transform_decimal(sgn * v)
            assert abs(got - want) <= 2e-15 * abs(want) + 1e-300, (v, got, want)


@pytest.mark.parametrize("delta", [0.1, 0.5, 1.0, 3.0])
@pytest.mark.parametrize("width", [1, 8, 9, 21, 51, 201, 255, 256])
def test_decode_bound_holds_for_the_kernel_arithmetic_and_not_for_its_mutations(width, delta):
    """A float32 emulation of the decode is within decode_ref's bound; the emulation with the final * delta dropped or
    with s0 = 1 + eps is outside it."""
    rng = np.random.default_rng(width)
    h = (width - 1) // 2
    support = (np.arange(width, dtype=np.float32) - np.float32(h)) * np.float32(delta)
    x = (rng.normal(0, 3, (24, width))).astype(np.float32)
    x[0] = 0
    x[1, -1] += 20
    x[2, 0] += 110
    x[3] *= 0.01
    out, bound = decode_ref(x, support, delta)
    emu = kernel_emulation(x, support, delta)
    assert (np.abs(emu - out) <= bound).all(), np.max(np.abs(emu - out) / np.maximum(bound, 1e-300))
    if width > 1:
        for kw in (dict(s0_one_eps=True),) + ((dict(drop_delta=True),) if delta != 1.0 else ()):
            bad = kernel_emulation(x, support, delta, **kw)
            assert (np.abs(bad - out) > bound).any(), kw


def test_search_config_rejects_searches_without_root_visits():
    """num_simulations - 1 simulations run: one simulation leaves no visit to pick a move or a target from."""
    from hanabizero_b200.mcts import SearchConfig
    for n in (0, 1):
        with pytest.raises(ValueError, match="num_simulations"):
            SearchConfig(num_simulations=n)
    assert SearchConfig(num_simulations=2).num_simulations == 2
