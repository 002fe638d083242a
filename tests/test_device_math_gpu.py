"""GPU: the library's device math run by itself over its whole domain.

- glibc's expf (hz_math.cuh), which every root and expanded prior goes through: expf_glibc and expf_glibc_warp on all
  2^32 float bit patterns against the glibc restatement oracle/expf_glibc.h (checked against libm by
  test_oracle_expf.py), bit for bit, any NaN for NaN.  The warp form runs twice: 32 consecutive patterns per warp, so
  every lane meets every table index, then 32 patterns 2^27 apart, so one warp mixes signs, magnitudes, inf / NaN and
  the |x| >= 88 fallback with the polynomial path.
- det_log / det_exp (hz_detmath.cuh), the float64 primitives of the root noise, on the device against the host build
  of the same source (tests/detmath_harness.cu), bit for bit: every binade for det_log, [-745, 0] and every switch of
  the reduction for det_exp.  test_device_math_cpu.py ties that host build to the float64 port of the noise.
- Root noise across the accepted alpha range [1e-300, 1e300] through the library's entry points: device == host twin
  bit for bit, no NaN, rows summing to 1."""
from decimal import Decimal

import numpy as np
import pytest
import torch

from helpers import build_detmath_harness, build_expf_check, det_exp_edges, det_exp_uniform, det_log_points, expf_check

pytestmark = pytest.mark.gpu

CHUNK = 1 << 26


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    return build_detmath_harness(tmp_path_factory.mktemp("detmath"))


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    return build_expf_check(tmp_path_factory.mktemp("expf_check"))


def _expf_sweep(harness, checker, warp_forms, rotate):
    """All 2^32 patterns, CHUNK at a time, through each form in warp_forms (0 = expf_glibc, 1 = expf_glibc_warp);
    every form of a chunk is checked against one evaluation of the reference.  -> [(mismatches, first patterns)]."""
    stream = torch.cuda.current_stream()
    dev = [torch.empty(CHUNK, dtype=torch.int32, device="cuda") for _ in warp_forms]
    host = [torch.empty(CHUNK, dtype=torch.int32, pin_memory=True) for _ in warp_forms]
    total = [(0, []) for _ in warp_forms]
    for start in range(0, 1 << 32, CHUNK):
        for w, d, h in zip(warp_forms, dev, host):
            assert harness.hzt_expf(stream.cuda_stream, d.data_ptr(), start, CHUNK, w, rotate) == 0
            h.copy_(d, non_blocking=True)
        stream.synchronize()
        got = expf_check(checker, [h.numpy().view(np.uint32) for h in host], start, rotate)
        total = [(n + m, (f + g)[:16]) for (n, f), (m, g) in zip(total, got)]
    return total


def _report(results):
    return {k: (n, [f"{p:#010x}" for p in first]) for k, (n, first) in results.items() if n}


def test_expf_matches_glibc_on_every_pattern(harness, checker):
    scalar, warp = _expf_sweep(harness, checker, (0, 1), rotate=0)
    bad = _report({"expf_glibc": scalar, "expf_glibc_warp": warp})
    assert not bad, bad


def test_expf_warp_matches_glibc_with_mixed_lanes(harness, checker):
    (warp,) = _expf_sweep(harness, checker, (1,), rotate=1)
    bad = _report({"expf_glibc_warp, lanes 2^27 apart": warp})
    assert not bad, bad


def _device_vs_host(harness, name, blocks):
    """det_log / det_exp of every block on the device and on the host: (points, mismatches, first mismatches)."""
    stream = torch.cuda.current_stream()
    points, bad, first = 0, 0, []
    for x in blocks:
        x = np.ascontiguousarray(x)
        xd = torch.from_numpy(x).cuda()
        yd = torch.empty_like(xd)
        assert getattr(harness, "hzt_" + name)(stream.cuda_stream, xd.data_ptr(), yd.data_ptr(), x.size) == 0
        yh = np.empty_like(x)
        getattr(harness, "hzt_host_" + name)(x.ctypes.data, yh.ctypes.data, x.size)
        y = yd.cpu().numpy()
        miss = np.flatnonzero(y.view(np.int64) != yh.view(np.int64))
        first += [(float(x[i]).hex(), float(y[i]).hex(), float(yh[i]).hex()) for i in miss[:8 - len(first)]]
        points, bad = points + x.size, bad + miss.size
    return points, bad, first


def test_det_log_device_equals_host_on_every_binade(harness):
    """2^16 random mantissas in each of the 2046 normal binades, plus each binade's mantissas 1, 1 + ulp, 2 - ulp
    and the 17 around the sqrt(2) split."""
    points, bad, first = _device_vs_host(harness, "det_log", det_log_points(1 << 16, seed=11))
    assert points == 2046 * ((1 << 16) + 20)
    assert bad == 0, (bad, first)


def test_det_exp_device_equals_host_on_its_domain(harness):
    """2^26 uniform points on [-745, 0]; +-8 ulps around -700, -580, +0 and -0; +-4 ulps around every switch of the
    reduction's k in [-1010, 0]."""
    blocks = [det_exp_edges()] + list(det_exp_uniform(1 << 26, seed=12))
    points, bad, first = _device_vs_host(harness, "det_exp", blocks)
    assert points == 2 * 17 + 18 + 1011 * 9 + (1 << 26)
    assert bad == 0, (bad, first)


# every half decade from 1e-300 to 1e300, and the two sides of the switch into the alpha < 1 boost path
GRID_ALPHAS = [float(Decimal(10) ** (Decimal(k) / 2)) for k in range(-600, 601)]
SPECIAL_ALPHAS = [1e-300, 1e300, float(np.nextafter(1.0, 0.0)), 1.0, float(np.nextafter(1.0, 2.0))]
NOISE_AS = (1, 2, 3, 20, 32)


def test_dirichlet_device_equals_host_across_the_alpha_range():
    """hz_dirichlet_noise == hz_host_dirichlet_noise bit for bit, 129 roots at each A, over the whole accepted alpha
    range; at the five special alphas also with the seed's high word and the step's top bit set."""
    from hanabizero_b200.selfplay import dirichlet_noise, dirichlet_noise_host
    assert GRID_ALPHAS[0] == 1e-300 and GRID_ALPHAS[-1] == 1e300 and GRID_ALPHAS[600] == 1.0
    cases = [(alpha, 0x2545F4914F6CDD1D, 3) for alpha in GRID_ALPHAS + SPECIAL_ALPHAS]
    cases += [(alpha, 0xC0FFEE0123456789, 0x9E3779B9) for alpha in SPECIAL_ALPHAS]
    failures = []
    for alpha, seed, step in cases:
        dev = [dirichlet_noise(129, A, alpha, "cuda", seed=seed, step=step) for A in NOISE_AS]
        for A, d in zip(NOISE_AS, dev):
            d = d.cpu().numpy()
            h = dirichlet_noise_host(129, A, alpha, seed=seed, step=step)
            if (d.view(np.uint32) != h.view(np.uint32)).any():
                failures.append(("device != host", alpha, A, seed, step))
            if np.isnan(d).any() or np.isnan(h).any():
                failures.append(("NaN", alpha, A, seed, step))
            if A > 1 and np.abs(d.astype(np.float64).sum(1) - 1.0).max() > 2.0 ** -24 * A:
                failures.append(("sum", alpha, A, seed, step))
    assert not failures, (len(failures), failures[:8])
