"""CPU: the host half of tests/detmath_harness.cu, and the expf checker of the device sweep.

test_device_math_gpu.py compares det_log / det_exp on the device with the harness's host build of hz_detmath.cuh.
Here that host build is checked bit for bit against the independent float64 port of test_noise_reference_cpu.py,
the reference that pins the library's own host twin, so "device == harness host" means "device == the twin".
The harness is built in full (nvcc cross-compiles the device half too); only its host functions run."""
import ctypes

import numpy as np
import pytest

from helpers import build_detmath_harness, build_expf_check, det_exp_edges, det_exp_uniform, det_log_points, expf_check
from test_noise_reference_cpu import det_exp as port_det_exp
from test_noise_reference_cpu import det_log as port_det_log
from test_noise_reference_cpu import fma as port_fma


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    return build_detmath_harness(tmp_path_factory.mktemp("detmath"))


def _host(fn, x):
    x = np.ascontiguousarray(x, np.float64)
    y = np.empty_like(x)
    fn(x.ctypes.data, y.ctypes.data, x.size)
    return y


def _assert_bits_equal(x, got, want):
    bad = np.flatnonzero(got.view(np.int64) != want.view(np.int64))
    assert bad.size == 0, (bad.size, [(float(x[i]).hex(), float(got[i]).hex(), float(want[i]).hex()) for i in bad[:4]])


def test_harness_host_det_log_equals_the_port(harness):
    """One random mantissa per binade, every binade, plus each binade's mantissas 1, 1 + ulp, 2 - ulp and the 17
    around the sqrt(2) split: 43 000 points."""
    x = next(det_log_points(1, block=2046, seed=5))
    assert x.size == 2046 * 21 and (x > 0).all() and np.isfinite(x).all() and (x >= 2.0 ** -1022).all()
    _assert_bits_equal(x, _host(harness.hzt_host_det_log, x), port_det_log(x))


def test_harness_host_det_exp_equals_the_port(harness):
    x = np.concatenate([det_exp_edges(), next(det_exp_uniform(4096, seed=6))])
    _assert_bits_equal(x, _host(harness.hzt_host_det_exp, x), port_det_exp(x))


def test_det_exp_edges_straddle_every_reduction_switch():
    """Each +-4 ulp window around (k - 1/2) ln 2 holds points reduced with k - 1 and with k, so the sweep meets the
    switch itself and not only its neighbourhood."""
    ks = np.arange(-1010, 1)
    x = det_exp_edges(ks)[-ks.size * 9:].reshape(ks.size, 9)
    kf = np.floor(port_fma(x, 1.44269504088896338700, 0.5))
    assert (kf.min(1) == ks - 1).all() and (kf.max(1) == ks).all()


# ---- the expf checker (tests/expf_check.c) -------------------------------------------------------------------------

def pattern(i, rotate):
    u = np.asarray(i, np.uint64).astype(np.uint32)
    return (u >> np.uint32(5)) | (u << np.uint32(27)) if rotate else u


@pytest.mark.parametrize("rotate", [0, 1])
def test_expf_checker_reports_exactly_the_mismatches(tmp_path, rotate):
    """libm's expf stands in for a device: the checker finds nothing on it, then exactly the entries changed, first
    ones first, and accepts a NaN of another payload for a NaN."""
    lib = build_expf_check(tmp_path)
    libm = ctypes.CDLL("libm.so.6")
    libm.expf.argtypes, libm.expf.restype = [ctypes.c_float], ctypes.c_float
    # unrotated: patterns around 1.0 (the polynomial path) and around inf (overflow, inf, NaN)
    for start in (0x3F800000 - (1 << 12), 0x7F800000 - (1 << 12)):
        p = pattern(start + np.arange(1 << 13), rotate)
        x = p.view(np.float32)
        y = np.array([libm.expf(float(v)) for v in x.tolist()], np.float32).view(np.uint32)
        assert expf_check(lib, [y], start, rotate) == [(0, [])]
        z = y.copy()
        nan = np.isnan(y.view(np.float32))
        z[nan] ^= np.uint32(0x80000001)   # another NaN: sign and payload are not part of the contract
        ok = np.flatnonzero(~nan)
        pick = ok[[3, ok.size // 2, ok.size - 2]]
        z[pick] ^= np.uint32(1)
        z[-1] = np.uint32(0) if nan[-1] else np.uint32(0x7FC00000)
        got = expf_check(lib, [y, z], start, rotate, nfirst=3)
        assert got[0] == (0, []) and got[1] == (4, p[pick].tolist()), (hex(start), got)
