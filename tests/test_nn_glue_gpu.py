"""GPU: the small network-side entry points of the C ABI against torch — hz_support_decode (inverse
categorical transform, core/config.py:210-232), hz_gemm_plan (cuBLASLt chain) and
hz_gather_hidden.  Float tolerance (these are floating-point glue around library GEMMs, not tree state)."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ref_decode(logits, support, delta=1.0, dtype=torch.float64):
    """core/config.py:210-232 (inverse_scalar_transform) written with torch ops as the reference writes it."""
    probs = torch.softmax(logits.to(dtype), dim=1)
    v = (probs * support.to(dtype)).sum(1) / delta
    eps = 0.001
    out = ((torch.sqrt(1 + 4 * eps * (v.abs() + 1 + eps)) - 1) / (2 * eps)) ** 2 - 1
    out = torch.where(v < 0, -out, out) * delta
    return torch.nan_to_num(out, nan=0.0)


# widths around the decode's 8-column lane segments (1, 7, 8, 9, 63, 64, 65), the Hanabi supports (21, 51, 201) and the
# limit (255, 256), in both dtypes; an ld that is not a multiple of 8 takes the scalar load path
DECODE_CASES = [(torch.float32, 201, 201), (torch.float16, 201, 208), (torch.float32, 51, 56)] + [
    (dt, w, ld) for w, lds in ((1, (1, 8)), (7, (8, 7)), (8, (8, 12)), (9, (9, 16)), (21, (24, 21)), (63, (63, 64)),
                               (64, (64, 68)), (65, (72, 65)), (255, (255, 256)), (256, (256, 264)))
    for dt, ld in zip((torch.float32, torch.float16), lds)]


@pytest.mark.parametrize("dtype,width,ld", DECODE_CASES)
def test_support_decode_matches_float64_reference(dtype, width, ld):
    """float32 arithmetic with one approximate step (exp as ex2.approx.ftz, 2 ulp; IEEE division and square root):
    within the path's 1e-5 relative bar of a float64 evaluation of the reference's formula, plus 2e-5 absolute per 100
    of the support's half-width (at least 2e-5) — two ulp of the exponential times the half-width, which is what float32
    softmax sums over the support can cancel to (tests/test_selfplay_glue_gpu.py holds the decode to a bound derived
    term by term) — and closer to float64 than the reference's own float32 evaluation, whose textbook form
    cancels twice near zero (where that form loses anything at all).  The same rows read from a base one element past
    a 16-byte boundary (the scalar load path) decode to the same bits."""
    from hanabizero_b200 import _lib
    lib = _lib.load()
    rows = 4000
    x = (torch.randn(rows, ld, device="cuda") * 3).to(dtype)
    x[5, :width] = float("nan")
    x[6, :width] = 0.0                      # symmetric support, uniform probabilities: exactly zero
    x[7:300, :width] *= 0.05                # near-uniform rows: expectations near zero (the cancellation-prone region)
    support = torch.arange(width, device="cuda", dtype=torch.float32) - (width - 1) // 2
    st = torch.cuda.current_stream().cuda_stream
    out = torch.empty(rows, device="cuda")
    _lib.check(lib.hz_support_decode(st, x.data_ptr(), x.element_size(), support.data_ptr(), out.data_ptr(), rows,
                                     width, ld, 1.0))
    ref64 = _ref_decode(x[:, :width], support)
    half = max(abs(support[0].item()), abs(support[-1].item()))
    torch.testing.assert_close(out.double(), ref64, rtol=1e-5, atol=2e-5 * max(1.0, half / 100))
    assert out[5].item() == 0.0 and (width % 2 == 0 or out[6].item() == 0.0)
    ref32 = _ref_decode(x[:, :width], support, dtype=torch.float32).double()
    ours, theirs = (out.double() - ref64).abs().max().item(), (ref32 - ref64).abs().max().item()
    assert ours < theirs or (theirs < 1e-9 and ours <= theirs), f"ours {ours:.2e} vs the float32 textbook form {theirs:.2e}"
    shifted = torch.empty(rows * ld + 1, device="cuda", dtype=dtype)
    shifted[1:].copy_(x.reshape(-1))
    out2 = torch.empty(rows, device="cuda")
    _lib.check(lib.hz_support_decode(st, shifted[1:].data_ptr(), x.element_size(), support.data_ptr(), out2.data_ptr(),
                                     rows, width, ld, 1.0))
    assert torch.equal(out2, out), "scalar and vector load paths disagree"


def test_support_decode_transform_is_ieee_exact_on_one_hot_rows():
    """One-hot logits make the expectation exactly a support point, so the output is the inverse transform alone:
    it must equal, bit for bit, the same cancellation-free formula evaluated with numpy float32 scalars (every
    operation correctly rounded — no ex2/rsqrt/fast-division approximations anywhere)."""
    from hanabizero_b200 import _lib
    lib = _lib.load()
    width, ld = 201, 208
    x = torch.full((width, ld), -30000.0, device="cuda", dtype=torch.float32)
    x[torch.arange(width), torch.arange(width)] = 0.0
    support = torch.arange(width, device="cuda", dtype=torch.float32) - 100
    out = torch.empty(width, device="cuda")
    _lib.check(lib.hz_support_decode(torch.cuda.current_stream().cuda_stream, x.data_ptr(), 4, support.data_ptr(),
                                     out.data_ptr(), width, width, ld, 1.0))
    f = np.float32
    v = np.arange(-100, 101).astype(np.float32)
    a = np.abs(v)
    eps = f(0.001)
    y = f(f(4.0) * eps) * ((a + f(1.0)) + eps)
    sq = np.sqrt(f(1.0) + y)
    u = (f(2.0) * a) / (sq + f(f(1.0) + f(f(2.0) * eps)))
    want = np.where(v < 0, -(u * (u + f(2.0))), u * (u + f(2.0))).astype(np.float32)
    got = out.cpu().numpy()
    assert (got.view(np.uint32) == want.view(np.uint32)).all() or (got == want).all()
    exact = _ref_decode(x[:, :width], support).cpu().numpy()
    np.testing.assert_allclose(got, exact, rtol=1e-6, atol=1e-9)   # (the float64 textbook form itself leaves 2e-15 at v = 0)


def test_gemm_plan_matches_torch_linear():
    from hanabizero_b200 import _lib
    from hanabizero_b200._lib import GemmStep
    lib = _lib.load()
    dev = torch.device("cuda")
    m, k, n = 300, 256, 208
    for dtype, tol in ((torch.float16, 2e-2), (torch.float32, 1e-4)):
        a = torch.randn(3, m, k, device=dev).to(dtype)
        w = (torch.randn(3, n, k, device=dev) * 0.05).to(dtype)
        b = torch.randn(3, n, device=dev).to(dtype)
        c = torch.randn(m, n, device=dev).to(dtype)
        d1 = torch.zeros(3, m, n, device=dev, dtype=dtype)
        d2 = torch.zeros(m, n, device=dev, dtype=dtype)
        s1, s2 = GemmStep(), GemmStep()
        s1.a, s1.lda, s1.stride_a = a.data_ptr(), k, m * k          # strided batch of 3, bias, ReLU
        s1.w, s1.ldw, s1.stride_w = w.data_ptr(), k, n * k
        s1.bias, s1.stride_bias = b.data_ptr(), n
        s1.d, s1.ldd, s1.stride_d = d1.data_ptr(), n, m * n
        s1.m, s1.n, s1.k, s1.batch, s1.relu = m, n, k, 3, 1
        s2.a, s2.lda = a[0].data_ptr(), k                           # single GEMM, bias + residual, no ReLU
        s2.w, s2.ldw = w[1].data_ptr(), k
        s2.bias = b[1].data_ptr()
        s2.c, s2.ldc = c.data_ptr(), n
        s2.d, s2.ldd = d2.data_ptr(), n
        s2.m, s2.n, s2.k, s2.batch, s2.relu = m, n, k, 1, 0
        h = ctypes.c_void_p()
        _lib.check(lib.hz_gemm_plan_create(ctypes.byref(h), 0, a.element_size(), (GemmStep * 2)(s1, s2), 2))
        assert lib.hz_gemm_plan_steps(h) == 2
        _lib.check(lib.hz_gemm_plan_run(h, torch.cuda.current_stream().cuda_stream, 0, 2))
        ref1 = torch.relu(torch.einsum("bmk,bnk->bmn", a.float(), w.float()) + b.float()[:, None, :])
        ref2 = a[0].float() @ w[1].float().t() + b[1].float() + c.float()
        torch.testing.assert_close(d1.float(), ref1, rtol=tol, atol=tol)
        torch.testing.assert_close(d2.float(), ref2, rtol=tol, atol=tol)
        _lib.check(lib.hz_gemm_plan_destroy(h))


def test_gather_hidden_standalone():
    from hanabizero_b200 import _lib
    lib = _lib.load()
    S, N, F = 7, 100, 512
    pool = torch.randn(S, N, F, device="cuda")
    ix = torch.randint(0, S, (N,), device="cuda", dtype=torch.int32)
    iy = torch.randperm(N, device="cuda").int()
    out = torch.empty(N, F, device="cuda")
    _lib.check(lib.hz_gather_hidden(torch.cuda.current_stream().cuda_stream, pool.data_ptr(), ix.data_ptr(), iy.data_ptr(),
                                    out.data_ptr(), N, F * 4))
    assert torch.equal(out, pool[ix.long(), iy.long()])


@pytest.mark.parametrize("n,target", [(512, 24), (96, 16), (2048, 56)])
def test_gemm_sm_target_keeps_the_function(n, target):
    """hz_gemm_plan_set_sm_target only changes WHICH library kernels run (sized for a share of the SMs, for searches in
    flight): the chain's outputs stay the same function — equal to the default kernels' within fp16 rounding — and
    setting the target back to 0 restores the default kernels' bits."""
    from hanabizero_b200.model import MuZeroNetFull
    from hanabizero_b200.plan import BoundChain
    dev = torch.device("cuda")
    torch.manual_seed(0)
    model = MuZeroNetFull(785 * 4, 20).randomize_heads().to(dev).eval()
    plan = model.recurrent_plan(torch.float16)
    ch = BoundChain(plan, n)
    gen = torch.Generator(device=dev).manual_seed(1)
    ch.x0.copy_(torch.rand(ch.x0.shape, device=dev, generator=gen).half())
    st = torch.cuda.current_stream().cuda_stream
    ch.run(st)
    base_out, base_state = ch.out.clone(), ch.state.clone()
    ch.set_sm_target(target)
    ch.run(st)
    torch.testing.assert_close(ch.out.float(), base_out.float(), rtol=2e-2, atol=4e-3)
    torch.testing.assert_close(ch.state.float(), base_state.float(), rtol=2e-2, atol=4e-3)
    ch.set_sm_target(0)
    ch.run(st)
    assert torch.equal(ch.out, base_out) and torch.equal(ch.state, base_state)
