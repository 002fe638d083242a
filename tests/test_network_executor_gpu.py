"""GPU: both executors of the recurrent plan (hanabizero_b200/plan.py) — the cuBLASLt chain ("library") and the
row-block resident kernel k_row_chain ("rows", hanabizero_b200/csrc/hz_rowchain.cu) — against ONE reference: a float64
copy of the nn.Module (copy.deepcopy(net).double().eval()) run through its dynamics and prediction networks.  The
reference is not the folded plan, so an error in the BatchNorm folding (RecurrentPlan.refresh), which both executors
share, shows here.  Covered: every shape the row executor accepts, row counts up to every CTA running 3-4 row blocks,
a recurrent unroll through a pool as the search runs it (eager and graph-replayed), and non-finite rows.

Tolerances, from fp16 arithmetic.  u = 2^-11 is the unit roundoff of fp16; both executors accumulate in fp32, whose
2^-24 per addition over K <= 544 terms is negligible next to it.
  * Every layer rounds its output to fp16 (<= u of the value) and multiplies by folded weights rounded to fp16 (<= u
    per product; the products' signs are random, so their sum is off by ~u of the output, not by u of sum |w x|).
  * Eval-mode BN keeps each layer's gain O(1), so the layers' errors add rather than multiply.
  A tensor L layers deep (DEPTH: s' 3; Hanabi-Full value / reward logits 6, policy 7; Hanabi-Small logits 5) is
  therefore within ~2 L u of its largest magnitude.  Asserted for the library chain against the module:
  4 L u max|reference| (1.4 % for the Hanabi-Full policy).  A BN bias left out of the folding shifts activations of
  magnitude ~1 by ~0.2, ten times that.
  * The row executor computes the same sums in another order: its error is asserted within 2x the library's plus
    u max|reference| (half an ulp of the largest value), as in tests/test_rowchain_gpu.py.
"""
import copy

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U = 2.0 ** -11
KEYS = ("state", "value", "reward", "policy")
DEPTH = {True: dict(state=3, value=6, reward=6, policy=7), False: dict(state=3, value=5, reward=5, policy=5)}
SENTINEL = -5.0          # never an output: s' >= 0 after its ReLU, padding columns are 0.0


class Cfg:
    pb_c_base, pb_c_init, discount, value_delta_max, num_simulations, amp_type = 19652, 1.25, 0.997, 0.01, 30, "torch_amp"


def _net(full, A, support, seed=1):
    """Non-trivial BN statistics and affine terms, output heads re-drawn (the reference zero-initialises them)."""
    from hanabizero_b200.model import MuZeroNet, MuZeroNetFull
    torch.manual_seed(seed)
    net = (MuZeroNetFull(785, A, support, support) if full else MuZeroNet(193, A, support, support))
    net = net.randomize_heads(std=0.05, seed=seed).to("cuda")
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.normal_(0, 0.2); m.running_var.uniform_(0.5, 1.5)
            m.weight.data.uniform_(0.5, 1.5); m.bias.data.normal_(0, 0.2)
    return net.eval()


def _actions(n, A, gen):
    """Random actions, except that rows 0..A-1 and 127-(A-1)..127 of every 128-row block take every action in turn."""
    a = torch.randint(0, A, (n,), device="cuda", generator=gen)
    r = torch.arange(n, device="cuda") % 128
    a = torch.where(r < A, r, a)
    return torch.where(r >= 128 - A, 127 - r, a)


def _fill(ch, plan, seed):
    """[hidden >= 0 | one-hot] as the tree kernel hands it over.  Edge rows: row 64 has no action column set, and the
    state columns 0..OH-1 of rows 65..70 are exactly 1.0 (a one-hot scan wider than the row's own OH columns would
    read one of them as an action)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    F, n = plan.F, ch.n
    ch.x0.zero_()
    ch.x0[:, :F] = (torch.randn(n, F, device="cuda", generator=g).clamp_min(0) * 0.7).half()
    ch.x0[:, F:].scatter_(1, _actions(n, plan.A, g)[:, None], 1.0)
    if n > 70:
        ch.x0[64, F:] = 0
        ch.x0[65:71, :plan.OH] = 1.0


def _reference(net64, x0, plan):
    """float64 module on the batch: dynamics() is _dynamics_state over [state | one-hot] then _dynamics_reward; the
    one-hot is the batch's own columns (zero for a row without an action).  Then prediction()."""
    x = x0.double()
    s = net64._dynamics_state(torch.cat((x[:, :plan.F], x[:, plan.F:plan.F + plan.A]), 1))
    reward = net64._dynamics_reward(s)
    policy, value = net64.prediction(s)
    return dict(state=s, value=value, reward=reward, policy=policy)


def _outputs(state, out, plan):
    W, A = plan.n_support, plan.A
    return dict(state=state, value=out[0, :, :W], reward=out[1, :, :W], policy=out[2, :, :A])


def _errors(ref, state, out, plan):
    got = _outputs(state, out, plan)
    return {k: (got[k].double() - ref[k]).abs().max().item() for k in KEYS}


def _padding_is_zero(out, plan, what):
    W, A = plan.n_support, plan.A
    for i, c in ((0, W), (1, W), (2, A)):
        assert torch.count_nonzero(out[i, :, c:]) == 0, f"{what}: padding columns {c}..{plan.P3} of output {i}"


def _assert_bounds(plan, ref, e_lib, e_rows, where=""):
    for k in KEYS:
        scale = max(ref[k].abs().max().item(), 1e-3)
        bound = 4 * DEPTH[plan.full][k] * U * scale
        assert e_lib[k] <= bound, f"{where}library {k}: {e_lib[k]:.3g} from the float64 module > {bound:.3g}"
        assert e_rows[k] <= 2 * e_lib[k] + U * scale, f"{where}rows {k}: {e_rows[k]:.3g} vs library {e_lib[k]:.3g}"


def _both_executors(plan, n, seed):
    """Library chain then row executor on the same BoundChain buffers (rows writes s' to a buffer of its own, as the
    search re-binds the state output to pool[x]).  Returns the chain and both executors' (s', out)."""
    from hanabizero_b200.plan import BoundChain
    ch = BoundChain(plan, n)
    assert ch.rows_supported()
    _fill(ch, plan, seed)
    st = torch.cuda.current_stream().cuda_stream
    ch.out.fill_(SENTINEL)
    ch.bind_state(ch.state)
    ch.run(st)
    s_lib, o_lib = ch.state.clone(), ch.out.clone()
    s_rows = torch.full_like(ch.state, SENTINEL)
    ch.out.fill_(SENTINEL)
    ch.set_executor("rows")
    ch.bind_state(s_rows)
    ch.run(st)
    torch.cuda.synchronize()
    assert torch.equal(ch.state, s_lib), "the row executor must leave the library's (unbound) state buffer alone"
    return ch, (s_lib, o_lib), (s_rows, ch.out.clone())


def _float64(net):
    """The reference module.  Copied before the module's plans exist (they own library handles, which must not be
    copied)."""
    assert "_plans" not in net.__dict__
    return copy.deepcopy(net).double().eval()


def _check_against_module(net, n, seed):
    net64 = _float64(net)
    plan = net.recurrent_plan(torch.float16)
    ch, (s_lib, o_lib), (s_rows, o_rows) = _both_executors(plan, n, seed)
    ref = _reference(net64, ch.x0, plan)
    _padding_is_zero(o_lib, plan, "library")
    _padding_is_zero(o_rows, plan, "rows")
    _assert_bounds(plan, ref, _errors(ref, s_lib, o_lib, plan), _errors(ref, s_rows, o_rows, plan))
    return plan


# (full, A, support, P3): every one-hot width and logit width the row executor accepts (BoundChain.rows_supported):
# Hanabi-Full 17..32 actions (32 one-hot columns: 20..31 only set from A = 21 on) with P3 from 32 (some epilogue warps
# own no logit columns) to 256 (the staged logits fill tile K-blocks 0..3 and 4..7 exactly); Hanabi-Small 1..16
# actions with 49..63 support logits (P3 = 64).  P3 = round_up(max(support, A), 16): (20, 15) has 20 policy logits.
SHAPES = [
    (True, 20, 201, 208), (True, 32, 255, 256), (True, 17, 21, 32), (True, 20, 15, 32), (True, 25, 41, 48),
    (True, 20, 101, 112),
    (False, 11, 51, 64), (False, 16, 63, 64), (False, 1, 49, 64),
]


@pytest.mark.parametrize("full,A,support,p3", SHAPES)
def test_executors_match_float64_module_at_every_accepted_shape(full, A, support, p3):
    """1000 rows (7 full row blocks and a partial one of 104 rows): every action at both ends of a block."""
    plan = _check_against_module(_net(full, A, support), 1000, seed=A * 1000 + support)
    assert (plan.full, plan.A, plan.n_support, plan.P3) == (full, A, support, p3)


# n = blocks * g * 128 + extra, g the device's SM count: around one and two row blocks, one full wave of CTAs, one row
# block more (one CTA runs two), and 3 g + 1 blocks (every CTA runs 3 or 4 row blocks: the grid-stride loop, the
# prefetch of the next block's s and the barrier parities carried across blocks, several times per CTA)
ROWS = [(0, 127), (0, 129), (0, 255), (0, 257), (1, 0), (1, 1), (3, 77)]


@pytest.mark.parametrize("full,blocks,extra", [(True,) + r for r in ROWS] + [(False, 0, 129), (False, 1, 1), (False, 3, 77)])
def test_executors_match_float64_module_across_row_counts(full, blocks, extra):
    g = torch.cuda.get_device_properties(0).multi_processor_count
    n = blocks * g * 128 + extra
    _check_against_module(_net(full, 20 if full else 11, 201 if full else 51, seed=2), n, seed=n)


def _unroll(ch, pool, acts, K, check=None):
    """What the search does: step k feeds pool[k-1] (with a fresh one-hot) and writes s' into pool[k] (bind_state)."""
    F = ch.plan.F
    st = torch.cuda.current_stream().cuda_stream
    for k in range(1, K + 1):
        ch.x0[:, :F].copy_(pool[k - 1])
        ch.x0[:, F:].zero_()
        ch.x0[:, F:].scatter_(1, acts[k][:, None], 1.0)
        ch.bind_state(pool[k])
        ch.run(st)
        if check is not None:
            check(k)


@pytest.mark.parametrize("full,graph", [(True, False), (False, False), (True, True)])
def test_recurrent_unroll_through_a_pool(full, graph):
    """K = 12 steps of n = 4096 + 77 rows, each executor feeding its own outputs back through its own pool, as the
    search does.  After every step: s' landed in pool[k] only (pool[k+1..K] keep their sentinel, pool[k-1] is
    unchanged); per-step error (the float64 module fed the step's own fp16 input) within the module bounds above,
    rows within 2x library + floor; error growth (the float64 module running its own float64 chain from pool[0]): rows
    within 2x library + floor at every k.  graph: the whole unroll captured in one CUDA graph per executor and replayed
    onto a fresh pool must reproduce the eager pool and outputs bit for bit."""
    from hanabizero_b200.plan import BoundChain
    K, n = 12, 4096 + 77
    A, support = (20, 201) if full else (11, 51)
    net = _net(full, A, support, seed=4)
    net64 = _float64(net)
    plan = net.recurrent_plan(torch.float16)
    gen = torch.Generator(device="cuda").manual_seed(7)
    acts = [None] + [_actions(n, A, gen) for _ in range(K)]
    s0 = (torch.randn(n, plan.F, device="cuda", generator=gen).clamp_min(0) * 0.7).half()
    chains, pools, steps = {}, {}, {}
    for ex in ("library", "rows"):
        ch = chains[ex] = BoundChain(plan, n)
        if ex == "rows":
            ch.set_executor("rows")
        pool = pools[ex] = torch.full((K + 1, n, plan.F), SENTINEL, dtype=torch.float16, device="cuda")
        pool[0] = s0
        steps[ex] = []

        def check(k, ch=ch, pool=pool, ex=ex):
            torch.cuda.synchronize()
            assert (pool[k + 1:] == SENTINEL).all(), f"{ex} step {k}: wrote past pool[{k}]"
            assert not (pool[k] == SENTINEL).any(), f"{ex} step {k}: rows of pool[{k}] not written"
            before = steps[ex][-1][0] if steps[ex] else s0
            assert torch.equal(pool[k - 1], before), f"{ex} step {k}: its input pool[{k - 1}] changed"
            steps[ex].append((pool[k].clone(), ch.out.clone(), ch.x0.clone()))

        _unroll(ch, pool, acts, K, check)
    s64 = s0.double()
    for k in range(1, K + 1):
        (s_lib, o_lib, x_lib), (s_rows, o_rows, x_rows) = steps["library"][k - 1], steps["rows"][k - 1]
        ref_lib, ref_rows = _reference(net64, x_lib, plan), _reference(net64, x_rows, plan)
        e_lib, e_rows = _errors(ref_lib, s_lib, o_lib, plan), _errors(ref_rows, s_rows, o_rows, plan)
        _assert_bounds(plan, ref_lib, e_lib, e_rows, f"step {k}: ")
        x64 = torch.cat((s64, x_lib[:, plan.F:].double()), 1)
        ref64 = _reference(net64, x64, plan)
        g_lib, g_rows = _errors(ref64, s_lib, o_lib, plan), _errors(ref64, s_rows, o_rows, plan)
        for key in KEYS:
            floor = U * ref64[key].abs().max().item()
            assert g_rows[key] <= 2 * g_lib[key] + floor, \
                f"step {k} {key}: growth rows {g_rows[key]:.3g} vs library {g_lib[key]:.3g}"
        s64 = ref64["state"]
    if graph:
        for ex, ch in chains.items():
            pool = torch.full_like(pools[ex], SENTINEL)
            pool[0] = s0
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                _unroll(ch, pool, acts, K)
            g.replay()
            torch.cuda.synchronize()
            assert torch.equal(pool, pools[ex]), f"{ex}: graph replay differs from the eager unroll"
            assert torch.equal(ch.out, steps[ex][-1][1]), f"{ex}: graph replay's last outputs differ"


# rows of the second 128-row block: (row, columns, value)
POISON = [(130, slice(5, 6), float("nan")), (131, slice(None), float("nan")), (140, slice(77, 78), float("inf")),
          (141, slice(None), float("inf")), (150, slice(300, 301), 65504.0), (151, slice(None), 65504.0)]


@pytest.mark.parametrize("full", [True, False])
def test_non_finite_rows_stay_in_their_rows(full):
    """NaN, +inf and 65504 (the largest fp16) in the hidden state of a few rows of one block.  For each executor every
    other row is bit-identical to its run without the poisoned rows, and on the poisoned rows both executors agree on
    which outputs are finite (the search's NaN handling, hz_search_io.sanitize_nan, was built on the library chain).
    What each executor does:
      library: cuBLASLt's ReLU epilogue keeps NaN.  A NaN in a row's state makes its s' and all its logits NaN.  An inf
               (or 65504 in every column, which overflows fc1) becomes +-inf products, NaN where the next layer sums
               them with both signs: again s' and all logits NaN.  65504 in one column leaves s' finite but for one
               inf column, and the heads' sums of inf products make every logit NaN.
      rows:    the same, since its ReLU is __hmax2_nan.  With __hmax2 (which returns the non-NaN operand) it used to
               turn NaN into 0: NaN rows came out finite, and inf rows came out with finite value / reward logits
               beside NaN policy logits.
    """
    from hanabizero_b200.plan import BoundChain
    n = 384
    A, support = (20, 201) if full else (11, 51)
    net = _net(full, A, support, seed=5)
    plan = net.recurrent_plan(torch.float16)
    rows_p = torch.tensor([r for r, _, _ in POISON], device="cuda")
    clean = torch.ones(n, dtype=torch.bool, device="cuda")
    clean[rows_p] = False
    res = {}
    for ex in ("library", "rows"):
        ch = BoundChain(plan, n)
        ch.set_executor(ex)
        st = torch.cuda.current_stream().cuda_stream
        runs = []
        for poison in (False, True):
            _fill(ch, plan, seed=3)
            if poison:
                for r, cols, v in POISON:
                    ch.x0[r, :plan.F][cols] = v
            ch.out.fill_(SENTINEL)
            ch.state.fill_(SENTINEL)
            ch.run(st)
            torch.cuda.synchronize()
            runs.append((ch.state.clone(), ch.out.clone()))
        (s0, o0), (s1, o1) = runs
        assert torch.equal(s1[clean], s0[clean]) and torch.equal(o1[:, clean], o0[:, clean]), f"{ex}: a clean row changed"
        _padding_is_zero(o1[:, clean], plan, ex)
        res[ex] = (s1[rows_p], o1[:, rows_p])
    (s_l, o_l), (s_r, o_r) = res["library"], res["rows"]
    assert torch.equal(torch.isfinite(s_l), torch.isfinite(s_r)), "s' of the poisoned rows: finite in one executor only"
    assert torch.equal(torch.isfinite(o_l), torch.isfinite(o_r)), "logits of the poisoned rows: finite in one executor only"


def _search_inputs(full, A, support, N, seed):
    from hanabizero_b200.model import MuZeroNet, MuZeroNetFull
    torch.manual_seed(0)
    inp = 785 if full else 193
    model = (MuZeroNetFull if full else MuZeroNet)(inp, A, support, support).randomize_heads(seed=0).to("cuda").eval()
    rng = np.random.default_rng(seed)
    obs = torch.from_numpy((rng.random((N, inp)) < 0.2).astype(np.float32)).cuda()
    with torch.no_grad():
        _, logits, hidden = model.initial_inference_device(obs)
    legal = torch.from_numpy((rng.random((N, A)) < 0.7).astype(np.int32)).cuda()
    legal[:, 0] = 1
    noise = torch.from_numpy(rng.dirichlet([0.3] * A, N).astype(np.float32)).cuda()
    return model, logits, hidden, legal, noise


def _search(cfg, model, logits, hidden, legal, noise, executor, repeats):
    from hanabizero_b200 import cytree
    from hanabizero_b200.mcts import MCTS
    N, A = legal.shape
    mcts = MCTS(cfg)
    for _ in range(repeats):     # eager, then capture + replay
        roots = cytree.Roots(N, A, cfg.num_simulations)
        roots.prepare(0.25, noise, torch.zeros(N, device="cuda"), logits.float(), legal)
        mcts.run_multi(roots, model, hidden, executor=executor)
    v, val = roots.get_stats_tensors()
    return mcts, v.clone(), val.clone()


def test_search_with_row_executor_at_32_actions_and_support_21():
    """A whole search on Hanabi-Full with 32 actions (one-hot columns 20..31 set) and a 21-wide support (the fused
    decode at width 21, P3 = 32): the assertions of tests/test_rowchain_gpu.py's search test — same visit totals, >= 0.99
    of the root actions identical, root values within 1e-2."""
    N, A, S = 1024, 32, Cfg.num_simulations
    inputs = _search_inputs(True, A, 21, N, 4)
    stats = {}
    for ex in ("library", "rows"):
        mcts, v, val = _search(Cfg, *inputs, ex, 3)
        assert all(ws.chain._use_rows == (ex == "rows") for ws in mcts._ws.values())
        stats[ex] = (v, val)
    (v0, val0), (v1, val1) = stats["library"], stats["rows"]
    assert int(v1.sum()) == N * (S - 1) and torch.equal(v0.sum(1), v1.sum(1))
    agree = (v0.argmax(1) == v1.argmax(1)).float().mean().item()
    assert agree >= 0.99, agree
    assert (val0 - val1).abs().max().item() < 1e-2


# (full, A, support, dtype, the tree step accepts the support)
REFUSED = [(True, 16, 201, torch.float16, True), (True, 20, 257, torch.float16, False),
           (False, 17, 51, torch.float16, True), (False, 11, 47, torch.float16, True),
           (False, 11, 65, torch.float16, True), (True, 20, 201, torch.float32, True)]


@pytest.mark.parametrize("full,A,support,dtype,tree_ok", REFUSED)
def test_refused_plans_stay_on_the_library_chain(full, A, support, dtype, tree_ok):
    """Plans outside the row executor's shapes (Hanabi-Full with <= 16 actions or a support over 255, Hanabi-Small with
    over 16 actions or a support outside 49..63, fp32): set_executor("rows") raises, and a search asked for the row
    executor runs the library chain — with the same visits as executor="library"."""
    from hanabizero_b200.plan import BoundChain
    net = _net(full, A, support)
    plan = net.recurrent_plan(dtype)
    ch = BoundChain(plan, 256)
    assert not ch.rows_supported()
    with pytest.raises(RuntimeError):
        ch.set_executor("rows")
    if not tree_ok:
        return
    cfg = type("C", (Cfg,), dict(num_simulations=10, amp_type="torch_amp" if dtype == torch.float16 else "none"))
    inputs = _search_inputs(full, A, support, 256, 6)
    visits = {}
    for ex in ("library", "rows"):
        mcts, v, _ = _search(cfg, *inputs, ex, 1)
        assert not any(ws.chain._use_rows for ws in mcts._ws.values())
        visits[ex] = v
    assert torch.equal(visits["library"], visits["rows"])
