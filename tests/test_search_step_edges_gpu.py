"""GPU: the fused tree step (hz_trees_search_step, k_search_step) in lock-step with the CPU oracle at the edges of its
compiled paths, with the generic calls (hz_support_decode + hz_trees_backprop_traverse, k_tree_step) run on the same
inputs beside it so that a failure names the kernel that diverged.

Each simulation x >= 1 writes raw network outputs into the kernel's input buffers with torch ops on the search's
stream (value / reward support rows and policy logits at a leading dimension wider than the row, pool[x] or the
`next_state` side buffer), then runs the step.  The oracle is fed hz_support_decode's values and rewards of the same
rows and the policy logits as float32 with NaN -> 0 and nothing else (what `sanitize_nan` does in both kernels).
Compared bit for bit (NaN payloads aside): root priors; per simulation the parent index and action, the hand-off row
(hidden state, one-hot columns, padding columns still holding a sentinel) and min/max after each back-propagation; at
the end visit counts, root values, path lengths, trajectories and every expanded node.

What the cases reach, in the kernel's terms:
  * A4 = ceil(A / 4) rounded to the instantiation: 3 (A <= 12), 5 (A <= 20), 8 (A <= 32);
  * capacity <= 254 reads pb_c from the per-(parent, child) `pbc` table, above it from `lut` plus a division;
    q is staged in shared memory while cap + 1 <= 1024 (rows of 4 floats);
  * level_eval_exact: a dividend outside [2^-87, 2^94) or a min-max span outside [2^-27, 2^34) (support scaled far
    from 1), each case checking from the oracle's own state that it really got there;
  * rows wider than 1 KB leave the two-register hand-off for warp_copy16."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import CONST, bits_equal, nan_to_zero, tree_inputs

pytestmark = pytest.mark.gpu

SENTINEL = -3.25   # exact in fp16 and fp32; batch columns the kernel must not write keep it


def _round_up(a, b):
    return (a + b - 1) // b * b


# ---- per-simulation network outputs: (gen, S, N, A, W) -> value [S,N,W], reward [S,N,W], policy [S,N,A], float32 ----
def randn_rows(gen, S, N, A, W):
    dev = gen.device
    return (torch.randn(S, N, W, device=dev, generator=gen), torch.randn(S, N, W, device=dev, generator=gen),
            torch.randn(S, N, A, device=dev, generator=gen))


def uniform_rows(gen, S, N, A, W):
    """Zero logits everywhere: uniform policies, and value / reward rows that decode to exactly 0 (odd width,
    symmetric support)."""
    dev = gen.device
    return torch.zeros(S, N, W, device=dev), torch.zeros(S, N, W, device=dev), torch.zeros(S, N, A, device=dev)


def nonfinite_rows(gen, S, N, A, W):
    """randn rows, and per (simulation, tree) a seeded choice of: policy rows with one NaN / +inf / -inf, all -inf,
    all NaN, +-65504 (the largest fp16), all equal; value rows all NaN, with one +inf, or uniform; reward rows with
    -inf entries, all -inf, or uniform."""
    v, r, p = randn_rows(gen, S, N, A, W)
    dev = gen.device
    nan, inf = float("nan"), float("inf")

    def kind(k):
        return torch.randint(0, k, (S, N), device=dev, generator=gen)

    def one_col(width):
        return torch.nn.functional.one_hot(torch.randint(0, width, (S, N), device=dev, generator=gen), width).bool()

    kp, ka = kind(10), one_col(A)
    p = torch.where((kp == 1)[..., None] & ka, nan, p)
    p = torch.where((kp == 2)[..., None] & ka, inf, p)
    p = torch.where((kp == 3)[..., None] & ka, -inf, p)
    p[kp == 4] = -inf
    p[kp == 5] = nan
    big = torch.where(torch.rand(S, N, A, device=dev, generator=gen) < 0.5, -65504.0, 65504.0)
    p = torch.where((kp == 6)[..., None], big, p)
    p[kp == 7] = 0.0
    kv, kw = kind(8), one_col(W)
    v[kv == 1] = nan
    v = torch.where((kv == 2)[..., None] & kw, inf, v)
    v[kv == 3] = 0.0
    kr = kind(8)
    some = torch.rand(S, N, W, device=dev, generator=gen) < 0.25
    r = torch.where((kr == 1)[..., None] & some, -inf, r)
    r[kr == 2] = -inf
    r[kr == 3] = 0.0
    return v, r, p


def make_inputs(N, A, S, W=201, F=512, dtype=torch.float16, seed=0, rows=randn_rows, mask_mode="random"):
    """Root inputs (helpers.tree_inputs) and the network outputs of every simulation, generated up front."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    v, r, p = rows(gen, S, N, A, W)
    pool = torch.rand(S + 1, N, F, device="cuda", generator=gen).to(dtype)   # pool[x]: what the network writes at x
    return dict(root=tree_inputs(N, A, S, seed, mask_mode), value=v.to(dtype), reward=r.to(dtype), policy=p.to(dtype),
                pool=pool)


def slice_inputs(inp, lo, hi):
    return dict(root={k: inp["root"][k][lo:hi] for k in ("logits", "noise", "reward", "mask")},
                value=inp["value"][:, lo:hi].contiguous(), reward=inp["reward"][:, lo:hi].contiguous(),
                policy=inp["policy"][:, lo:hi].contiguous(), pool=inp["pool"][:, lo:hi].contiguous())


def _bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def lockstep(inp, cap=None, support_scale=1.0, support_delta=1.0, delta=CONST["delta"], discount=CONST["discount"],
             pb_c_base=CONST["pb_c_base"], pb_c_init=CONST["pb_c_init"], tie=None, tree_offset=0, stage_limit=0,
             onehot_cols=None, ld_batch=None, noise=True, next_state=False, programmatic=False):
    """Run the fused step, the generic calls and the oracle through the same search; assert that all three agree.

    cap: tree capacity (max_sims of hz_trees_create); default S + 1, what cytree.Roots(N, A, S) allocates.  The search
    runs S simulations: traverses at x = 0 .. S-2, back-propagations at x = 1 .. S-1 (the last without a traverse).
    Returns the oracle's and the fused step's records for case-specific checks."""
    from hanabizero_b200 import _lib, cytree
    from oracle import loader as L
    lib = _lib.load()
    dev = torch.device("cuda")
    st = torch.cuda.current_stream().cuda_stream
    S, N, W = inp["value"].shape
    A, F = inp["policy"].shape[2], inp["pool"].shape[2]
    dtype = inp["pool"].dtype
    eb = inp["pool"].element_size()
    cap = S + 1 if cap is None else cap
    assert S - 1 <= cap
    OH = _round_up(A, 16) if onehot_cols is None else onehot_cols
    LDB = F + _round_up(A, 16) + 8 if ld_batch is None else ld_batch
    d = inp["root"]
    nz = d["noise"] if noise else None
    rows = torch.arange(N, device=dev)
    support = (torch.arange(W, device=dev, dtype=torch.float32) - (W - 1) // 2) * support_scale

    # raw rows as the kernel reads them: leading dimension wider than the row, NaN in the columns past it
    LD, LDP = _round_up(W, 8) + 8, _round_up(A, 8) + 8
    raw = torch.full((S, 2, N, LD), float("nan"), device=dev, dtype=dtype)
    raw[:, 0, :, :W] = inp["value"]
    raw[:, 1, :, :W] = inp["reward"]
    dec = torch.empty(S, 2, N, device=dev)
    _lib.check(lib.hz_support_decode(st, raw.data_ptr(), eb, support.data_ptr(), dec.data_ptr(), S * 2 * N, W, LD,
                                     support_delta))

    def new_roots():
        roots = cytree.Roots(N, A, cap - 1)
        if tie is not None:
            roots.set_tie_break("random", tie, tree_offset)
        if noise:
            roots.prepare(CONST["frac"], d["noise"], d["reward"], d["logits"], d["mask"])
        else:
            roots.prepare_no_noise(d["reward"], d["logits"], d["mask"])
        mm = cytree.MinMaxStatsList(N)
        mm.set_delta(delta)
        return roots, mm.tensor(dev)

    def finish(roots):
        v, val = roots.get_stats_tensors()
        e = roots.export(cap)
        return dict(visits=v.cpu().numpy(), values=val.cpu().numpy(), ex_reward=e["reward"].cpu().numpy(),
                    ex_value_sum=e["value_sum"].cpu().numpy(), ex_visits=e["visits"].cpu().numpy(),
                    plen=e["path_len"].cpu().numpy(), traj=roots.get_trajectories())

    def record_traverse(rec, x, ix, la):
        rec["ix"][x].copy_(ix)
        rec["la"][x].copy_(la)

    def new_record():
        return dict(ix=torch.full((S, N), -1, dtype=torch.int32, device=dev),
                    la=torch.full((S, N), -1, dtype=torch.int32, device=dev),
                    mm=torch.zeros(S, N, 2, device=dev), bad=torch.zeros(S, 3, dtype=torch.bool, device=dev))

    # ---- fused step: hz_trees_search_step on raw outputs ----
    roots_f, mm_f = new_roots()
    priors_f = roots_f.export(1)["root_priors"].cpu().numpy()
    pool = torch.zeros(S + 1, N, F, device=dev, dtype=dtype)
    pool[0] = inp["pool"][0]
    vr = torch.full((2, N, LD), float("nan"), device=dev, dtype=dtype)
    pol = torch.full((N, LDP), float("nan"), device=dev, dtype=dtype)
    state = torch.full((N, F + 8), SENTINEL, device=dev, dtype=dtype) if next_state else None
    batch = torch.full((N, LDB), SENTINEL, device=dev, dtype=dtype)
    ix = torch.zeros(N, dtype=torch.int32, device=dev)
    la = torch.zeros(N, dtype=torch.int32, device=dev)
    io = _lib.SearchIO()
    io.value_logits, io.ld_value = vr[0].data_ptr(), LD
    io.reward_logits, io.ld_reward = vr[1].data_ptr(), LD
    io.policy_logits, io.ld_policy = pol.data_ptr(), LDP
    io.next_state, io.ld_state = (state.data_ptr(), F + 8) if next_state else (None, 0)
    io.support, io.support_width, io.support_delta = support.data_ptr(), W, support_delta
    io.elem_bytes, io.sanitize_nan = eb, 1
    io.pool, io.state_cols = pool.data_ptr(), F
    io.out_batch, io.ld_batch, io.onehot_cols = batch.data_ptr(), LDB, OH
    io.out_ix, io.out_action = ix.data_ptr(), la.data_ptr()
    io.minmax, io.value_delta_max = mm_f.data_ptr(), delta
    io.discount, io.pb_c_base, io.pb_c_init = discount, pb_c_base, pb_c_init
    io.programmatic_launch, io.stage_limit = int(programmatic), stage_limit
    ref = ctypes.byref(io)
    fused = new_record()
    want_pad = torch.full((N, LDB - F - OH), SENTINEL, device=dev, dtype=dtype)
    for x in range(S):
        if x >= 1:
            (state[:, :F] if next_state else pool[x]).copy_(inp["pool"][x])
            vr.copy_(raw[x])
            pol[:, :A].copy_(inp["policy"][x])   # a kernel (strided destination): the step's programmatic predecessor
        _lib.check(lib.hz_trees_search_step(roots_f.handle, st, x, int(x < S - 1), ref))
        if x >= 1:
            fused["mm"][x].copy_(mm_f)
        if x < S - 1:
            record_traverse(fused, x, ix, la)
            want = inp["pool"][ix.long(), rows]
            fused["bad"][x, 0].copy_((_bits(batch[:, :F]) != _bits(want)).any())
            onehot = torch.zeros(N, OH, device=dev, dtype=dtype)
            if OH:
                onehot[rows, la.long()] = 1.0
            fused["bad"][x, 1].copy_((_bits(batch[:, F:F + OH]) != _bits(onehot)).any())
            fused["bad"][x, 2].copy_((_bits(batch[:, F + OH:]) != _bits(want_pad)).any())
    fused_end = finish(roots_f)
    assert torch.equal(_bits(pool[1:S]), _bits(inp["pool"][1:S])), "pool[x] after the search"

    # ---- generic calls: decoded values + hz_trees_backprop_traverse with the gather ----
    roots_g, mm_g = new_roots()
    priors_g = roots_g.export(1)["root_priors"].cpu().numpy()
    hidden = torch.zeros(N, F, device=dev, dtype=dtype)
    generic = new_record()
    src = inp["pool"]
    for x in range(S):
        if x == 0:
            _lib.check(lib.hz_trees_traverse(roots_g.handle, st, pb_c_base, pb_c_init, discount, mm_g.data_ptr(), delta,
                                             ix.data_ptr(), None, la.data_ptr(), None, src.data_ptr(), hidden.data_ptr(),
                                             F * eb))
        else:
            logits = inp["policy"][x].float().contiguous()
            args = (roots_g.handle, st, x, discount, dec[x, 1].data_ptr(), dec[x, 0].data_ptr(), logits.data_ptr(), 1,
                    mm_g.data_ptr())
            if x < S - 1:
                _lib.check(lib.hz_trees_backprop_traverse(*args, delta, pb_c_base, pb_c_init, ix.data_ptr(), None,
                                                          la.data_ptr(), None, src.data_ptr(), hidden.data_ptr(), F * eb))
            else:
                _lib.check(lib.hz_trees_backprop(*args))
            generic["mm"][x].copy_(mm_g)
        if x < S - 1:
            record_traverse(generic, x, ix, la)
            generic["bad"][x, 0].copy_((_bits(hidden) != _bits(src[ix.long(), rows])).any())
    generic_end = finish(roots_g)

    # ---- the oracle on the decoded values and NaN -> 0 logits ----
    h_dec = dec.cpu().numpy()
    h_pol = inp["policy"].float().cpu().numpy()
    cpu = L.oracle_tree(N, A, cap, delta)
    if tie is not None:
        cpu.set_tie(1, tie, tree_offset)
    cpu.prepare(CONST["frac"], nz, d["reward"], d["logits"], d["mask"])
    o = dict(priors=cpu.root_priors(), ix=np.full((S, N), -1, np.int32), la=np.full((S, N), -1, np.int32),
             mm=np.zeros((S, N, 2), np.float32))
    for x in range(S):
        if x >= 1:
            cpu.backprop(x, discount, h_dec[x, 1], h_dec[x, 0], nan_to_zero(h_pol[x]))
            o["mm"][x] = cpu.stats()[2]
        if x < S - 1:
            o["ix"][x], _, o["la"][x] = cpu.traverse(pb_c_base, pb_c_init, discount)
    o["visits"], o["values"], _ = cpu.stats()
    o["plen"] = cpu.path_lens()
    otr = cpu.trajectories(cap + 1)
    o["traj"] = [row[row >= 0].tolist() for row in otr]
    o["ex_reward"], o["ex_value_sum"] = np.zeros((N, cap), np.float32), np.zeros((N, cap), np.float32)
    o["ex_visits"] = np.zeros((N, cap), np.int32)
    for i in range(N):
        r, vs, vc = cpu.expanded_stats(i, cap)
        assert len(r) == S - 1
        o["ex_reward"][i, :S - 1], o["ex_value_sum"][i, :S - 1], o["ex_visits"][i, :S - 1] = r, vs, vc

    # ---- compare: the first divergence of each kernel ----
    errors = {}
    for name, priors, rec, end in (("k_search_step", priors_f, fused, fused_end),
                                   ("k_tree_step", priors_g, generic, generic_end)):
        rec = {k: v.cpu().numpy() for k, v in rec.items()}
        err = None if bits_equal(priors, o["priors"]) else "root priors"
        for x in range(S):
            if err:
                break
            if x < S - 1:
                for k in ("ix", "la"):
                    if (rec[k][x] != o[k][x]).any():
                        err = f"{k} at simulation {x}: trees {np.flatnonzero(rec[k][x] != o[k][x])[:8]}"
                        break
                if not err and rec["bad"][x].any():
                    part = ("hidden row", "one-hot columns", "padding columns")[int(np.argmax(rec["bad"][x]))]
                    err = f"hand-off {part} at simulation {x}"
            if not err and x >= 1 and not bits_equal(rec["mm"][x], o["mm"][x]):
                bad = [t for t in range(N) if not bits_equal(rec["mm"][x, t], o["mm"][x, t])]
                err = f"min/max after back-propagation {x}: trees {bad[:8]}"
        if not err:
            for k in ("visits", "values", "plen", "ex_reward", "ex_value_sum", "ex_visits"):
                if not bits_equal(end[k], o[k]):
                    err = k
                    break
        if not err and end["traj"] != o["traj"]:
            err = "trajectories"
        if err:
            errors[name] = err
    assert not errors, f"diverged from the oracle: {errors}"
    return dict(oracle=o, la=fused["la"].cpu().numpy(), delta=delta)


def reaches_exact_range(r):
    """From the oracle's state: some dividend of the traverse (a node's value sum or mean value) lies outside
    [2^-87, 2^94), or some normalising span (max(max - min, value_delta_max)) outside [2^-27, 2^34)."""
    o = r["oracle"]
    vs, vc = o["ex_value_sum"], o["ex_visits"]
    with np.errstate(all="ignore"):
        q = np.where(vc > 0, vs / np.maximum(vc, 1).astype(np.float32), 0).astype(np.float32)
        a = np.abs(np.concatenate([vs.ravel(), q.ravel()]))
        a = a[a != 0]
        dividend = bool(((a < 2.0 ** -87) | ~(a < 2.0 ** 94)).any())
        span = (o["mm"][1:, :, 1] - o["mm"][1:, :, 0]).astype(np.float32)
        span = span[span > 0]
        denom = np.where(span < r["delta"], np.float32(r["delta"]), span)
        extreme_span = bool(((denom < 2.0 ** -27) | ~(denom < 2.0 ** 34)).any())
    return dividend, extreme_span


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,A", [(torch.float16, a) for a in (1, 2, 3, 4, 5, 8, 11, 12, 13, 16, 17, 20, 21, 24, 31, 32)] +
                         [(torch.float32, a) for a in (1, 12, 13, 21, 32)])
def test_every_action_count(dtype, A):
    """Each A4 instantiation (3: A <= 12, 5: A <= 20, 8: A <= 32) on both sides of its bounds, and the one-hot width
    16 / 32 switch at A = 16 / 17."""
    lockstep(make_inputs(37, A, 40, dtype=dtype, seed=100 + A))


@pytest.mark.parametrize("limit", [0, 1, 4])
def test_32_actions_full_batch_partially_staged(limit):
    """4096 trees x 50 simulations at A = 32: 512-byte child records, so only part of each tree fits the shared-memory
    region (limit 0), or at most 1 / 4 staged nodes and q in global memory (hz_search_io.stage_limit)."""
    lockstep(make_inputs(4096, 32, 50, seed=7), stage_limit=limit)


@pytest.mark.parametrize("A", [3, 20, 32])
def test_one_traverse_then_back_propagation_only(A):
    lockstep(make_inputs(37, A, 2, seed=200 + A))


@pytest.mark.parametrize("A", [3, 20, 32])
@pytest.mark.parametrize("cap", [254, 255, 256, 1023, 1024, 1025])
def test_capacity_switches(cap, A):
    """pb_c from the `pbc` table (capacity <= 254) or from `lut` (above); q staged in shared memory (capacity + 1 <=
    1024) or read from global memory.  The search fills the capacity to its last slot."""
    lockstep(make_inputs(8, A, cap + 1, W=51, seed=cap + A), cap=cap)


@pytest.mark.parametrize("N,A", [(2, 3), (5, 20), (8, 32)])
def test_capacity_4100(N, A):
    r = lockstep(make_inputs(N, A, 4100, W=51, seed=N), cap=4100)
    assert r["oracle"]["visits"].sum() == N * 4099


@pytest.mark.parametrize("scale,delta,support_delta,dtype", [
    (1e-30, 0.006, 1.0, torch.float16),      # value sums below 2^-87
    (1e26, 0.006, 1.0, torch.float16),       # value sums above 2^94, spans above 2^34
    (1e30, 0.006, 1.0, torch.float32),
    (1e35, 0.006, 1.0, torch.float16),       # decoded values overflow to +-inf
    (1e-12, 1e-20, 1.0, torch.float16),      # spans below 2^-27 with value_delta_max below them
    (1e-30, 0.006, 0.5, torch.float32),
    (1e26, 0.006, 3.0, torch.float16),
])
def test_extreme_values_take_the_exact_division(scale, delta, support_delta, dtype):
    """Values far from 1 send whole traverse levels through level_eval_exact (a dividend outside div_safe's range)
    or every level (denom_ok false).  Asserted from the oracle's own state, so that the case cannot drift back to
    the branch-free path and pass for nothing."""
    r = lockstep(make_inputs(37, 20, 40, dtype=dtype, seed=300), support_scale=scale, delta=delta,
                 support_delta=support_delta)
    dividend, span = reaches_exact_range(r)
    assert dividend or span
    if scale == 1e-12:
        assert span
    if scale == 1e35:
        assert not np.isfinite(r["oracle"]["ex_value_sum"]).all()


@pytest.mark.parametrize("support_delta", [0.5, 3.0])
def test_support_delta(support_delta):
    lockstep(make_inputs(37, 20, 40, seed=310), support_delta=support_delta)


@pytest.mark.parametrize("dtype,A", [(torch.float16, 20), (torch.float16, 11), (torch.float32, 20), (torch.float32, 32)])
def test_nonfinite_raw_outputs(dtype, A):
    """NaN / +-inf / fp16-extreme logits straight from the network; the step zeroes NaN policy logits only, exactly
    what the oracle is given."""
    inp = make_inputs(37, A, 40, dtype=dtype, seed=400 + A, rows=nonfinite_rows)
    assert torch.isinf(inp["policy"]).any() and torch.isnan(inp["policy"]).any()
    lockstep(inp)


@pytest.mark.parametrize("A", [11, 20, 32])
def test_degenerate_ties(A):
    """Zero-initialised heads: uniform priors and zero values make every select an A-way tie.  Tie mode 0 takes the
    first index; tie mode 1 matches the oracle's generator, and a shard (tree_offset) draws what the full batch draws."""
    N, S = 64, 40
    inp = make_inputs(N, A, S, seed=500 + A, rows=uniform_rows)
    for k in ("logits", "reward"):
        inp["root"][k][:] = 0.0
    inp["root"]["mask"][:] = 1
    first = lockstep(inp, noise=False)
    assert (first["la"][0] == 0).all()
    full = lockstep(inp, noise=False, tie=99, tree_offset=7)
    assert len(np.unique(full["la"][0])) > A // 2
    lo, hi = 24, 56
    shard = lockstep(slice_inputs(inp, lo, hi), noise=False, tie=99, tree_offset=7 + lo)
    assert (shard["la"] == full["la"][:, lo:hi]).all()
    assert (shard["oracle"]["visits"] == full["oracle"]["visits"][lo:hi]).all()


@pytest.mark.parametrize("noise,mask_mode", [(True, "zero_rows"), (False, "zero_rows"), (False, "random")])
def test_roots(noise, mask_mode):
    """Every third root with an all-zero legal mask (the padding rows of a partial search wave), with and without
    noise; prepare_no_noise."""
    lockstep(make_inputs(48, 20, 40, seed=600, mask_mode=mask_mode), noise=noise)


@pytest.mark.parametrize("discount,pb_c_base,pb_c_init,delta", [
    (1.0, 19652, 1.25, 0.006), (0.997, 1, 1.25, 0.0), (1.0, 1, 0.0, 1e6), (0.997, 19652, 0.0, 0.006),
    (0.997, 19652, 1.25, 1e6),
])
def test_search_constants(discount, pb_c_base, pb_c_init, delta):
    lockstep(make_inputs(37, 20, 40, seed=700), discount=discount, pb_c_base=pb_c_base, pb_c_init=pb_c_init,
             delta=delta)


@pytest.mark.parametrize("dtype,F", [(torch.float16, 8), (torch.float16, 256), (torch.float16, 512),
                                     (torch.float16, 520), (torch.float32, 4), (torch.float32, 256),
                                     (torch.float32, 512)])
def test_hand_off_row_widths(dtype, F):
    """State rows of 16 bytes to 2 KB (two 16-byte registers per lane up to 1 KB, warp_copy16 above), with 8 padding
    columns after the one-hot block that must keep their sentinel."""
    lockstep(make_inputs(37, 20, 40, F=F, dtype=dtype, seed=800 + F))


def test_hand_off_from_next_state():
    """The network writes the new hidden state to a side buffer; the step copies it into pool[x]."""
    lockstep(make_inputs(37, 20, 40, seed=900), next_state=True)


def test_programmatic_launch():
    """programmatic_launch = 1 with a torch kernel writing the network outputs right before every step."""
    lockstep(make_inputs(37, 20, 40, seed=901), programmatic=True)


@pytest.mark.parametrize("A,onehot_cols", [(20, 20), (20, 32), (11, 11), (11, 16), (20, 0), (32, 0)])
def test_onehot_columns(A, onehot_cols):
    """onehot_cols >= A writes one-hot(action) over onehot_cols columns; 0 writes no column (all keep the sentinel)."""
    lockstep(make_inputs(37, A, 12, seed=1000 + A), onehot_cols=onehot_cols)


@pytest.mark.parametrize("A,onehot_cols", [(20, 1), (20, 16), (20, 19), (11, 8), (32, 31)])
def test_onehot_columns_short_of_the_actions_are_rejected(A, onehot_cols):
    from hanabizero_b200 import _lib, cytree
    lib = _lib.load()
    dev = torch.device("cuda")
    N, F = 4, 512
    roots = cytree.Roots(N, A, 8)
    roots.prepare_no_noise(np.zeros(N, np.float32), np.zeros((N, A), np.float32), np.ones((N, A), np.int32))
    mmt = cytree.MinMaxStatsList(N).tensor(dev)
    pool = torch.zeros(10, N, F, device=dev, dtype=torch.float16)
    batch = torch.full((N, F + 32), SENTINEL, device=dev, dtype=torch.float16)
    io = _lib.SearchIO()
    io.elem_bytes, io.pool, io.state_cols, io.out_batch, io.ld_batch = 2, pool.data_ptr(), F, batch.data_ptr(), F + 32
    io.minmax, io.value_delta_max, io.discount, io.pb_c_base, io.pb_c_init = mmt.data_ptr(), 0.006, 0.999, 19652, 1.25
    io.onehot_cols = onehot_cols
    st = torch.cuda.current_stream().cuda_stream
    assert lib.hz_trees_search_step(roots.handle, st, 0, 1, ctypes.byref(io)) == _lib.HZ_ERR_ARG
    assert b"onehot_cols" in lib.hz_last_error()
    assert (batch == SENTINEL).all()          # nothing was launched
    io.onehot_cols = A
    _lib.check(lib.hz_trees_search_step(roots.handle, st, 0, 1, ctypes.byref(io)))
    assert (batch[:, F:F + A].float().sum(1) == 1).all()
