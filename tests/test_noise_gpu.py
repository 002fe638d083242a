"""GPU: the device root noise (hz_dirichlet_noise) equals its host twin bit for bit at every action count, at the
4-warp blocks' tails, at the counters' edges, under each mask rule and on a non-default stream; its marginals follow
the float32-rounded Beta law at millions of rows; and neighbouring streams are uncorrelated.  The host twin itself is
checked against an independent float64 port and the Random123 known answers in test_noise_reference_cpu.py."""
import numpy as np
import pytest
import torch

from helpers import rounded_beta_ks

pytestmark = pytest.mark.gpu

ALPHAS = [1e-3, 0.03, 0.3, 0.999, 1.0, 1.5, 40.0]
COUNTERS = [(1234567890123, 0, 0), (0xDEADBEEF12345678, 2 ** 32 - 1, 7), (0xFFFFFFFF00000001, 99, 2 ** 32 - 3)]


@pytest.mark.parametrize("alpha", ALPHAS)
def test_device_dirichlet_equals_its_host_twin_bit_for_bit(alpha):
    """hz_dirichlet_noise (device) == hz_host_dirichlet_noise (host): same Philox streams, same IEEE float64
    arithmetic, so a device search can be replayed on the CPU with exactly its noise (SURVEY §8f N1)."""
    from hanabizero_b200.selfplay import dirichlet_noise, dirichlet_noise_host
    dev = torch.device("cuda")
    side = torch.cuda.Stream(dev)
    rng = np.random.default_rng(int(alpha * 1000) + 5)
    mask_values = np.array([0.0, -0.0, 0.5, np.nan, 1.0], np.float32)
    case = 0
    for A in range(1, 33):
        for N in (1, 3, 4, 5, 4097):
            seed, step, off = COUNTERS[case % len(COUNTERS)]
            legal = rng.choice(mask_values, (N, A)) if case % 2 else None
            stream = side if case % 3 == 0 else torch.cuda.current_stream(dev)
            with torch.cuda.stream(stream):
                lg = None if legal is None else torch.from_numpy(legal).to(dev)
                d = dirichlet_noise(N, A, alpha, dev, seed=seed, step=step, root_offset=off, legal=lg)
                plain = dirichlet_noise(N, A, alpha, dev, seed=seed, step=step, root_offset=off)
            stream.synchronize()
            d, plain = d.cpu().numpy(), plain.cpu().numpy()
            h = dirichlet_noise_host(N, A, alpha, seed=seed, step=step, root_offset=off, legal=legal)
            assert (d.view(np.uint32) == h.view(np.uint32)).all(), (A, N, seed, step, off)
            assert np.isfinite(plain).all() and (plain >= 0).all()
            np.testing.assert_allclose(plain.astype(np.float64).sum(1), 1.0, rtol=0, atol=2.0 ** -24 + 1e-12)
            # the mask zeroes entries whose value == 0 (-0 included) and leaves the others, 0.5 and NaN too, as drawn
            want = plain if legal is None else np.where(legal == 0.0, np.float32(0.0), plain)
            assert (d.view(np.uint32) == want.view(np.uint32)).all(), (A, N)
            case += 1


@pytest.mark.parametrize("A", [2, 3, 20])
@pytest.mark.parametrize("alpha", [0.01, 0.3, 1.5, 7.0])
def test_device_marginals_follow_the_rounded_beta_law(alpha, A):
    from hanabizero_b200.selfplay import dirichlet_noise
    n = 4 * 1024 * 1024
    x = dirichlet_noise(n, A, alpha, "cuda", seed=31 + A, step=int(alpha * 100)).cpu().numpy()
    assert np.isfinite(x).all()
    for a in (0, A - 1):
        p = rounded_beta_ks(x[:, a], alpha, (A - 1) * alpha)
        assert p >= 1e-6, (a, p)


def test_neighbouring_streams_are_uncorrelated():
    """Component 0 of rows whose streams differ only in root (adjacent root_offset), step or seed (low and high
    word): every correlation within 5 standard errors of 0."""
    from hanabizero_b200.selfplay import dirichlet_noise
    n, A, alpha, seed, step = 1 << 20, 20, 0.3, 0x0123456789ABCDEF, 41
    draw = lambda **kw: dirichlet_noise(n, A, alpha, "cuda", **{"seed": seed, "step": step, **kw})[:, 0].double()
    base = draw()
    pairs = {"root": (base[0::2], base[1::2]),
             "step": (base, draw(step=step + 1)),
             "seed": (base, draw(seed=seed + 1)),
             "seed high word": (base, draw(seed=seed + (1 << 32)))}
    for name, (u, v) in pairs.items():
        r = float(torch.corrcoef(torch.stack((u, v)))[0, 1])
        assert abs(r) < 5.0 / np.sqrt(u.numel()), (name, r)
