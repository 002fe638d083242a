"""CPU: the root-noise generator (hz_noise.cu, run through its host twin hz_host_dirichlet_noise) against references
that do not share its source.

- Philox4x32-10: a Python port checked against Random123's known-answer vectors.
- The whole draw: an independent float64 port (Philox, uniform53, det_log / det_exp, the polar normal, Marsaglia-Tsang
  with the alpha < 1 boost and the small-alpha rescale, the ascending sum, one rounding to float32) that must equal
  the library bit for bit, over cases that reach every accept / reject branch and over rows that sit on float32
  rounding ties, where an error of 1e-13 in the float64 arithmetic shows.
- The distribution: every marginal of Dirichlet(alpha * 1_A) is Beta(alpha, (A - 1) alpha), and the library returns
  it rounded to float32, so each marginal is tested against that rounded law (KS), plus the covariance.
- Small alpha: no NaN rows, sums of 1, A = 1 gives exactly 1.0; the argument checks; a pin of the alpha 0.3 / 1.5
  streams so that the engines' noise never changes silently."""
import hashlib
import math
from fractions import Fraction

import numpy as np
import pytest

from hanabizero_b200 import _lib
from hanabizero_b200.selfplay import dirichlet_noise_host
from helpers import rounded_beta_ks

M32 = 0xFFFFFFFF
U64 = np.uint64

# ---- Philox4x32-10 (Salmon et al., SC'11), vectorised over uint64 arrays holding 32-bit words ---------------------


def philox4x32_10(ctr, key):
    c0, c1, c2, c3 = (np.asarray(w, np.uint64) for w in ctr)
    k0, k1 = (np.asarray(w, np.uint64) for w in key)
    for _ in range(10):
        p0, p1 = U64(0xD2511F53) * c0, U64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> U64(32)) ^ c1 ^ k0, p1 & U64(M32), (p0 >> U64(32)) ^ c3 ^ k1, p0 & U64(M32)
        k0, k1 = (k0 + U64(0x9E3779B9)) & U64(M32), (k1 + U64(0xBB67AE85)) & U64(M32)
    return c0, c1, c2, c3


# Random123 kat_vectors, philox4x32 10 rounds: (counter, key, output)
PHILOX_KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((M32,) * 4, (M32,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


def test_philox_port_gives_random123_known_answers():
    for ctr, key, want in PHILOX_KAT:
        got = tuple(int(w) for w in philox4x32_10(ctr, key))
        assert got == want, ([hex(w) for w in got], [hex(w) for w in want])


# ---- float64 arithmetic: a correctly rounded fma, vectorised ------------------------------------------------------
# Python 3.12 has no math.fma.  a * b is split exactly into uh + ul (Veltkamp / Dekker), c + uh exactly into th + tl
# (Knuth's two-sum), and RN(th + RO(tl + ul)), with RO rounding to odd, is RN(a * b + c) (Boldo & Melquiond, "Emulation
# of FMA and correctly rounded sums: proved algorithms using rounding to odd", IEEE TC 57(4), 2008).  Exact as long
# as nothing over- or underflows, which holds for every operand below; test_fma_is_correctly_rounded checks it.

def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _split(x):
    t = 134217729.0 * x   # 2^27 + 1
    hi = t - (t - x)
    return hi, x - hi


def _two_prod(a, b):
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def _round_odd_sum(a, b):
    s, e = _two_sum(a, b)
    # consecutive doubles of one sign have consecutive bit patterns: when the sum is inexact and s is even, the odd
    # neighbour on the side of the exact value is the round-to-odd result
    fix = (e != 0) & ((s.view(np.int64) & 1) == 0)
    return np.where(fix, np.nextafter(s, np.where(e > 0, np.inf, -np.inf)), s)


def fma(a, b, c):
    a, b, c = (np.asarray(v, np.float64) for v in np.broadcast_arrays(a, b, c))
    uh, ul = _two_prod(a, b)
    th, tl = _two_sum(c, uh)
    return th + _round_odd_sum(tl, ul)


def _fma_exact(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def test_fma_is_correctly_rounded():
    rng = np.random.default_rng(0)
    n = 20000
    a = rng.standard_normal(n) * np.exp2(rng.integers(-60, 60, n))
    b = rng.standard_normal(n) * np.exp2(rng.integers(-60, 60, n))
    c = rng.standard_normal(n) * np.exp2(rng.integers(-120, 120, n))
    # ties and near-ties of a * b + c: c cancels the leading bits of the product
    c[: n // 4] = -(a[: n // 4] * b[: n // 4])
    c[n // 4: n // 2] = -np.nextafter(a[n // 4: n // 2] * b[n // 4: n // 2], 0.0)
    c[n // 2: n // 2 + 100] = 1.0
    a[n // 2: n // 2 + 100], b[n // 2: n // 2 + 100] = 1.0 + 2.0 ** -27, 2.0 ** -26   # exact half-ulp of 1
    got = fma(a, b, c)
    want = np.array([_fma_exact(x, y, z) for x, y, z in zip(a.tolist(), b.tolist(), c.tolist())])
    assert (got.view(np.int64) == want.view(np.int64)).all()


# ---- det_log / det_exp: the fixed polynomials of hz_noise.cu --------------------------------------------------------
LN2 = 0.69314718055994528623
SQRT2 = 1.4142135623730951


def det_log(x):
    """log x for normal x > 0: x = m 2^e with m in (sqrt(1/2), sqrt(2)], log m = 2 atanh(s), s = (m - 1) / (m + 1),
    the atanh series to s^23 in Horner form with fma, plus e log 2."""
    m, e = np.frexp(np.asarray(x, np.float64))
    m, e = m * 2.0, e - 1
    big = m > SQRT2
    m, e = np.where(big, m * 0.5, m), np.where(big, e + 1, e)
    s = (m - 1.0) / (m + 1.0)
    z = s * s
    p = np.full_like(s, 2.0 / 23.0)
    for k in (21, 19, 17, 15, 13, 11, 9, 7, 5, 3):
        p = fma(p, z, 2.0 / k)
    p = fma(p, z, 2.0)
    return fma(e.astype(np.float64), LN2, s * p)


def det_exp(x):
    """exp x for x <= 0, 0 below -700: x = k log 2 + r (log 2 split in two parts), the Taylor series of e^r to r^13
    with fma, then k added to the exponent."""
    x = np.asarray(x, np.float64)
    cut = x < -700.0
    x = np.where(cut, 0.0, x)
    kf = np.floor(fma(x, 1.44269504088896338700, 0.5))
    r = fma(kf, -0.693147180369123816490, x)
    r = fma(kf, -1.90821492927058770002e-10, r)
    p = np.full_like(r, 1.0 / 6227020800.0)
    for f in (479001600, 39916800, 3628800, 362880, 40320, 5040, 720, 120, 24, 6):
        p = fma(p, r, 1.0 / f)
    p = fma(p, r, 0.5)
    p = fma(p, r, 1.0)
    p = fma(p, r, 1.0)
    return np.where(cut, 0.0, np.ldexp(p, kf.astype(np.int64)))


def _ulps(got, want):
    return np.abs(got - want) / np.spacing(np.abs(want))


def test_det_log_is_accurate_to_a_few_ulp():
    rng = np.random.default_rng(1)
    n = 1_000_000
    parts = [np.ldexp(1.0 + rng.random(n), rng.integers(-1022, 1024, n)),      # every binade of the normals
             SQRT2 * (1.0 + (rng.random(20000) - 0.5) * 2.0 ** -40),            # both sides of the sqrt(2) split
             np.ldexp(SQRT2 * (1.0 + (rng.random(20000) - 0.5) * 2.0 ** -40), rng.integers(-1021, 1023, 20000)),
             1.0 + (rng.random(40000) - 0.5) * np.exp2(-rng.integers(1, 52, 40000)),   # x near 1: log x near 0
             np.array([SQRT2, np.nextafter(SQRT2, 0.0), np.nextafter(SQRT2, 2.0), 1.0, np.nextafter(1.0, 0.0),
                       np.nextafter(1.0, 2.0), 2.0 ** -1022, np.finfo(np.float64).max])]
    x = np.concatenate(parts)
    want = np.array([math.log(v) for v in x.tolist()])
    got = det_log(x)
    assert (got[x == 1.0] == 0.0).all()
    nz = want != 0.0
    assert _ulps(got[nz], want[nz]).max() <= 3.0
    assert (np.abs(got - want) <= 4.5e-16 * np.abs(want)).all()


def test_det_exp_is_accurate_to_a_few_ulp():
    rng = np.random.default_rng(2)
    n = 1_000_000
    k = np.arange(-1009, 1)
    parts = [-700.0 * rng.random(n),
             -np.exp2(-rng.integers(1, 60, 20000) * rng.random(20000)) * rng.random(20000),   # x near 0
             np.repeat(k * LN2, 10) * (1.0 + (rng.random(k.size * 10) - 0.5) * 2.0 ** -45),   # reduction boundaries
             (np.repeat(k, 10) + 0.5) * LN2,
             np.array([0.0, -0.0, -700.0, np.nextafter(-700.0, 0.0), -5e-324])]
    x = np.concatenate(parts)
    x = x[(x <= 0.0) & (x >= -700.0)]
    want = np.array([math.exp(v) for v in x.tolist()])
    got = det_exp(x)
    assert _ulps(got, want).max() <= 3.0
    assert (np.abs(got - want) <= 4.5e-16 * want).all()
    assert (det_exp(np.array([-700.0000001, -1e300, -np.inf])) == 0.0).all()


# ---- the whole draw -------------------------------------------------------------------------------------------------

def uniform53(hi, lo):
    """53 random bits -> (k + 1/2) 2^-53, strictly inside (0, 1), exact."""
    k = ((hi << U64(32)) | lo) >> U64(11)
    return (k.astype(np.float64) + 0.5) * 2.0 ** -53


BRANCHES = ("attempts>=3", "reject s>=1", "reject v<=0", "reject log", "accept squeeze", "accept log", "rescaled row")


def gamma_port(alpha, seed, step, root, action, branches):
    """Gamma(alpha, 1) for each stream (seed, step, root[i], action[i]); returns (g, log g) with log g = -inf for
    alpha >= 1.  Attempt t draws Philox blocks 2t and 2t + 1 of counter (block, action, root, step), key (seed lo,
    seed hi); block 2t gives the polar normal, block 2t + 1 the acceptance uniform and, for alpha < 1, U of
    Gamma(alpha + 1) * U^(1/alpha) (Marsaglia & Tsang 2000)."""
    n = root.size
    key = (seed & M32, seed >> 32)
    boost = alpha < 1.0
    a = alpha + 1.0 if boost else alpha
    d = a - 1.0 / 3.0
    c = 1.0 / math.sqrt(9.0 * d)
    g, lg = np.full(n, np.nan), np.full(n, -np.inf)
    todo = np.arange(n)
    t = 0
    while todo.size:
        m = todo.size
        ctr = lambda blk: (np.full(m, blk, np.uint64), action[todo], root[todo], np.full(m, step, np.uint64))
        b0, b1 = philox4x32_10(ctr(2 * t), key), philox4x32_10(ctr(2 * t + 1), key)
        v1 = 2.0 * uniform53(b0[0], b0[1]) - 1.0   # exact
        v2 = 2.0 * uniform53(b0[2], b0[3]) - 1.0
        s = fma(v1, v1, v2 * v2)
        in_disc = (s < 1.0) & (s != 0.0)
        s = np.where(in_disc, s, 0.5)
        x = v1 * np.sqrt((-2.0 * det_log(s)) / s)
        v = fma(c, x, 1.0)
        pos = in_disc & (v > 0.0)
        v = np.where(pos, v, 1.0)
        v = (v * v) * v
        u = uniform53(b1[0], b1[1])
        x2 = x * x
        squeeze = u < fma(-0.0331, x2 * x2, 1.0)
        log_test = det_log(u) < fma(0.5, x2, d * ((1.0 - v) + det_log(v)))
        accept = pos & (squeeze | log_test)
        branches["reject s>=1"] += int((~in_disc).sum())
        branches["reject v<=0"] += int((in_disc & ~pos).sum())
        branches["accept squeeze"] += int((pos & squeeze).sum())
        branches["accept log"] += int((pos & ~squeeze & log_test).sum())
        branches["reject log"] += int((pos & ~squeeze & ~log_test).sum())
        if t >= 2:
            branches["attempts>=3"] += int(accept.sum())
        gg = d * v
        if boost:
            e = det_log(uniform53(b1[2], b1[3])) / alpha
            lg[todo[accept]] = (det_log(gg) + e)[accept]
            gg = gg * det_exp(e)
        g[todo[accept]] = gg[accept]
        todo = todo[~accept]
        t += 1
    return g, lg


def dirichlet_port_f64(num, A, alpha, seed, step, root_offset=0, branches=None):
    """Gammas of streams (seed, step, root_offset + n mod 2^32, a), divided by their sum taken in ascending action
    order, in float64.  For alpha < 1 a row whose largest log-gamma m is below -580 uses exp(lg - m) instead."""
    branches = {b: 0 for b in BRANCHES} if branches is None else branches
    root = np.repeat((root_offset + np.arange(num, dtype=np.uint64)) & U64(M32), A)
    action = np.tile(np.arange(A, dtype=np.uint64), num)
    g, lg = gamma_port(alpha, seed, step & M32, root, action, branches)
    g, lg = g.reshape(num, A), lg.reshape(num, A)
    if alpha < 1.0:
        m = lg.max(1, keepdims=True)
        g = np.where(m < -580.0, det_exp(lg - m), g)
        branches["rescaled row"] += int((m < -580.0).sum())
    total = np.zeros(num)
    for a in range(A):
        total = total + g[:, a]
    return g / total[:, None]


def dirichlet_port(num, A, alpha, seed, step, root_offset=0, legal=None, branches=None):
    """dirichlet_port_f64 rounded once to float32; entries whose mask value == 0 are zeroed afterwards."""
    x = dirichlet_port_f64(num, A, alpha, seed, step, root_offset, branches).astype(np.float32)
    if legal is not None:
        x[legal == 0.0] = 0.0
    return x


def float32_tie_distance(q):
    """Relative distance of float64 values q > 0 from the nearest boundary between two float32 roundings."""
    f = q.astype(np.float32)
    lo = (f.astype(np.float64) + np.nextafter(f, np.float32(0)).astype(np.float64)) / 2
    hi = (f.astype(np.float64) + np.nextafter(f, np.float32(np.inf)).astype(np.float64)) / 2
    return np.minimum(np.abs(q - lo), np.abs(hi - q)) / q


PORT_ALPHAS = [1e-3, 0.03, 0.3, 0.999, 1.0, 1.5, 40.0]
PORT_AS = [1, 2, 7, 20, 32]


def _port_cases(alpha):
    """(num, A, seed, step, root_offset, legal) per A: plain counters, the seed's high word set with step 2^32 - 1,
    root_offset wrapping past 2^32, and a mask holding 0, -0, 0.5, NaN and 1."""
    rng = np.random.default_rng(int(alpha * 1e6) + 17)
    for A in PORT_AS:
        legal = rng.choice(np.array([0.0, -0.0, 0.5, np.nan, 1.0], np.float32), (48, A))
        yield 48, A, 5, 0, 0, None
        yield 48, A, 0xDEADBEEF12345678, 2 ** 32 - 1, 7, None
        yield 48, A, 0xFFFFFFFF00000001, 123456, 2 ** 32 - 24, legal


@pytest.mark.parametrize("alpha", PORT_ALPHAS)
def test_float64_port_equals_the_library_bit_for_bit(alpha):
    for num, A, seed, step, off, legal in _port_cases(alpha):
        want = dirichlet_port(num, A, alpha, seed, step, off, legal)
        got = dirichlet_noise_host(num, A, alpha, seed=seed, step=step, root_offset=off, legal=legal)
        bad = np.argwhere(got.view(np.uint32) != want.view(np.uint32))
        assert bad.size == 0, (A, seed, step, off, bad[:4].tolist(), got[tuple(bad[0])], want[tuple(bad[0])])


# Rows of (alpha 0.3, A 20, seed 0x9E3779B97F4A7C15, step 11) whose float64 quotient for the given action lies within
# 2e-14 of a float32 rounding boundary (found by scanning 200 000 rows with the port).  Ordinary rows round away any
# error below ~1e-8, so they cannot tell a det_log that is off by 1e-13 from a correct one; these rows can.
NEAR_TIES = [(38682, 8), (53799, 16), (182482, 0)]


def test_near_tie_rows_equal_the_port():
    seed, step, A = 0x9E3779B97F4A7C15, 11, 20
    for root, a in NEAR_TIES:
        q = dirichlet_port_f64(1, A, 0.3, seed, step, root)
        assert float32_tie_distance(q[0, a]) < 2e-14
        got = dirichlet_noise_host(1, A, 0.3, seed=seed, step=step, root_offset=root)
        assert (got.view(np.uint32) == q.astype(np.float32).view(np.uint32)).all(), (root, a)


def test_port_cases_reach_every_branch():
    branches = {b: 0 for b in BRANCHES}
    for alpha in PORT_ALPHAS:
        for num, A, seed, step, off, legal in _port_cases(alpha):
            dirichlet_port(num, A, alpha, seed, step, off, legal, branches)
    assert all(branches[b] > 0 for b in BRANCHES), branches


# ---- distribution: marginals against the float32-rounded Beta law ---------------------------------------------------

DIST_ALPHAS = [0.003, 0.01, 0.03, 0.3, 0.999, 1.0, 1.5, 7.0, 300.0]
DIST_AS = [2, 3, 11, 20, 32]


@pytest.mark.parametrize("A", DIST_AS)
@pytest.mark.parametrize("alpha", DIST_ALPHAS)
def test_marginals_follow_the_rounded_beta_law(alpha, A):
    n = 400_000 if A <= 3 else 200_000
    x = dirichlet_noise_host(n, A, alpha, seed=1000 + A, step=int(alpha * 1000) + 1)
    assert np.isfinite(x).all()
    for a in (0, A - 1):
        p = rounded_beta_ks(x[:, a], alpha, (A - 1) * alpha)
        assert p >= 1e-6, (a, p)
    # Cov(X_0, X_{A-1}) = -1 / (A^2 (A alpha + 1)); standard error from 100 batch means
    mu = 1.0 / A
    prod = ((x[:, 0].astype(np.float64) - mu) * (x[:, A - 1].astype(np.float64) - mu)).reshape(100, -1).mean(1)
    want = -1.0 / (A * A * (A * alpha + 1.0))
    z = (prod.mean() - want) / (prod.std(ddof=1) / 10.0)
    assert abs(z) < 4.9, (prod.mean(), want, z)


@pytest.mark.parametrize("alpha", [1e-300, 1e-4, 1e-3, 0.003, 0.01, 0.3, 1.0, 7.0, 300.0, 1e300])
def test_a_single_action_gets_exactly_one(alpha):
    x = dirichlet_noise_host(10000, 1, alpha, seed=0xABCDEF0123, step=4)
    assert (x == 1.0).all()


@pytest.mark.parametrize("alpha", [1e-300, 1e-6, 1e-4, 1e-3, 0.003, 0.01, 1e300])
@pytest.mark.parametrize("A", [2, 5, 20, 32])
def test_small_alpha_rows_are_finite_and_sum_to_one(alpha, A):
    n = 100_000 if alpha >= 1e-4 and A <= 5 else 20_000
    x = dirichlet_noise_host(n, A, alpha, seed=77, step=A)
    assert not np.isnan(x).any() and (x >= 0.0).all()
    # each of the A roundings to float32 is within 2^-24 of its (float64) value, relative
    assert np.abs(x.astype(np.float64).sum(1) - 1.0).max() <= 2.0 ** -24 + 1e-12


# ---- stream pin and argument checks ----------------------------------------------------------------------------------

def test_engine_streams_are_pinned():
    """SHA-256 of the alpha 0.3 and 1.5 streams as the generator drew them before the small-alpha rescale existed:
    any change to the Philox counters, the gamma draw or the normalisation shows here."""
    a = dirichlet_noise_host(4096, 20, 0.3, seed=0x9E3779B97F4A7C15, step=5, root_offset=0)
    b = dirichlet_noise_host(512, 11, 1.5, seed=7, step=2 ** 32 - 1, root_offset=2 ** 32 - 100)
    assert hashlib.sha256(a.tobytes()).hexdigest() == "a6e45bfec9029cd0adbec26e63ec2fe74ffc0c77b067bdf3c56253c16bbcae29"
    assert hashlib.sha256(b.tobytes()).hexdigest() == "e32b1831cac226b3d13bf3dc52cc38fc4e05888bc8620e40044515702845bb26"


BAD_ARGS = ([(1, 4, alpha) for alpha in (0.0, -0.0, -1.0, math.nan, math.inf, -math.inf, 9e-301, 2e300)] +
            [(1, 0, 0.3), (1, 33, 0.3), (0, 4, 0.3), (-1, 4, 0.3)])


@pytest.mark.parametrize("num,A,alpha", BAD_ARGS)
def test_bad_arguments_are_rejected_before_any_work(num, A, alpha):
    lib = _lib.load()
    out = np.full(64, 7.0, np.float32)
    assert lib.hz_host_dirichlet_noise(out.ctypes.data, num, A, alpha, 1, 0, 0, None) == _lib.HZ_ERR_ARG
    # the device entry point checks before it launches, so a host buffer and no stream never reach the GPU
    assert lib.hz_dirichlet_noise(None, out.ctypes.data, num, A, alpha, 1, 0, 0, None) == _lib.HZ_ERR_ARG
    assert (out == 7.0).all()
