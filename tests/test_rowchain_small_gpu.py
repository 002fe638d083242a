"""GPU: the row-block resident network executor on the Hanabi-Small network (MuZeroNet, hz_rowchain_create_small)
computes the same recurrent_inference as its five-launch cuBLASLt chain, in the search, in SearchPipeline and in
SelfPlayPool.  Floating point (fp16 storage, fp32 accumulation): the tolerance is stated per assertion; the tree step
that consumes these outputs stays bit-exact given its inputs."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

A = 11


class Cfg:
    pb_c_base, pb_c_init, discount, value_delta_max, num_simulations, amp_type = 19652, 1.25, 0.997, 0.01, 30, "torch_amp"


def _net(seed=1):
    from hanabizero_b200.model import MuZeroNet
    torch.manual_seed(seed)
    net = MuZeroNet(193 * 4, A).randomize_heads(std=0.05).to("cuda")
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.normal_(0, 0.2); m.running_var.uniform_(0.5, 1.5)
            m.weight.data.uniform_(0.5, 1.5); m.bias.data.normal_(0, 0.2)
    return net.eval()


def _fill(ch, plan, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    ch.x0.zero_()
    ch.x0[:, :plan.F].copy_((torch.randn(ch.n, plan.F, device="cuda", generator=g).clamp_min(0) * 0.7).half())
    a = torch.randint(0, plan.A, (ch.n, 1), device="cuda", generator=g)
    ch.x0[:, plan.F:].scatter_(1, a, 1.0)


def _ref64(ch, plan):
    """float64 evaluation of the plan's folded weights: relu(W1 [s|a] + b1 + s) -> fc2 -> fc3 -> heads."""
    w = {k: v.double() for k, v in plan._w.items()}
    x, H, relu = ch.x0.double(), plan.H, torch.relu
    y1 = relu(x @ w["W1"].T + w["b1"] + x[:, :plan.F]); y2 = relu(y1 @ w["W2"].T + w["b2"])
    s = relu(y2 @ w["W3"].T + w["b3"])
    h1 = relu(s @ w["Wh1"].T + w["bh1"])
    return s, torch.stack([h1[:, i * H:(i + 1) * H] @ w["WB3"][i].T + w["bB3"][i] for i in range(3)])


@pytest.mark.parametrize("n", [1, 128, 300, 1000, 4096, 19000])
def test_small_row_executor_matches_library_chain(n):
    """Every output of the one-launch executor against the library chain on the same buffers: row counts below, at and
    across the 128-row block size, one CTA looping over several row blocks (19000 rows > 148 blocks), a row without an
    action, and rows whose first state columns are exactly 1.0 (a one-hot scan wider than the 16 action columns of the
    row before them would take one of those for its action).  Both round fp32 sums to fp16 after every layer; they
    differ by summation order only, and both sit equally close to float64."""
    from hanabizero_b200.plan import BoundChain
    net = _net()
    plan = net.recurrent_plan(torch.float16)
    ch = BoundChain(plan, n)
    assert (plan.full, plan.H, plan.OH, plan.P3) == (False, 128, 16, 64) and ch.rows_supported()
    _fill(ch, plan, 5 + n)
    if n >= 300:
        ch.x0[7, plan.F:] = 0                      # no action column set: fc1 sees the state alone
        ch.x0[8:40:3, :16] = 1.0                   # rows 8, 11, ...: state columns 0..15 exactly 1.0
        ch.x0[8:40:3, plan.F:] = 0                 # ... of rows with one action each, not the first columns' index
        ch.x0[8:40:3, plan.F + 9] = 1.0
        ch.x0[9, plan.F:] = 0                      # the row after one of them has no action at all
        ch.x0[10, :16] = 1.0
    elif n > 1:
        ch.x0[1:, :16] = 1.0
    st = torch.cuda.current_stream().cuda_stream
    ch.bind_state(ch.state)
    ch.run(st)
    s_lib, o_lib = ch.state.clone(), ch.out.clone()
    other = torch.zeros_like(ch.state)
    ch.out.zero_()
    ch.set_executor("rows")
    ch.bind_state(other)                           # the search loop re-points the state output at pool[x]
    ch.run(st)
    torch.cuda.synchronize()
    assert torch.count_nonzero(ch.state - s_lib) == 0, "the unbound state buffer must be left alone"
    # <= 2 fp16 ulp of the largest activation, and never below the 3e-3 the Hanabi-Full test allows
    ulp = 2.0 ** (np.floor(np.log2(max(s_lib.abs().max().item(), 1e-3))) - 10)
    torch.testing.assert_close(other.float(), s_lib.float(), rtol=0, atol=max(3e-3, 2 * ulp))
    torch.testing.assert_close(ch.out.float(), o_lib.float(), rtol=0, atol=1e-3)
    s64, o64 = _ref64(ch, plan)
    e_rows, e_lib = (ch.out.double() - o64).abs().max().item(), (o_lib.double() - o64).abs().max().item()
    assert e_rows <= 2 * e_lib + 1e-4, (e_rows, e_lib)
    s_rows, s_l = (other.double() - s64).abs().max().item(), (s_lib.double() - s64).abs().max().item()
    assert s_rows <= 2 * s_l + 1e-3, (s_rows, s_l)
    ch.set_executor("library")
    ch.bind_state(ch.state)
    ch.state.zero_()
    ch.run(st)
    torch.cuda.synchronize()
    assert torch.equal(ch.state, s_lib)


def test_small_row_executor_follows_weight_updates_and_graph_replay():
    """The executor reads the plan's fixed weight buffers: refresh() after a parameter update is seen without
    re-creating anything, also by a CUDA graph captured before the update."""
    from hanabizero_b200.plan import BoundChain
    net = _net(seed=3)
    plan = net.recurrent_plan(torch.float16)
    ch = BoundChain(plan, 384)
    _fill(ch, plan, 9)
    ch.set_executor("rows")
    ch.bind_state(ch.state)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        ch.run(side.cuda_stream)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        ch.run(torch.cuda.current_stream().cuda_stream)
    g.replay(); torch.cuda.synchronize()
    before = ch.out.clone()
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(1.05)
    assert plan.refresh()
    g.replay(); torch.cuda.synchronize()
    after_rows = ch.out.clone()
    assert not torch.equal(before, after_rows)
    ch.set_executor("library")
    ch.run(torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    torch.testing.assert_close(after_rows.float(), ch.out.float(), rtol=0, atol=1e-3)


def _roots_inputs(N, seed):
    from hanabizero_b200.model import MuZeroNet
    torch.manual_seed(0)
    model = MuZeroNet(193 * 4, A).randomize_heads(seed=0).to("cuda").eval()
    rng = np.random.default_rng(seed)
    obs = torch.from_numpy((rng.random((N, 193 * 4)) < 0.2).astype(np.float32)).cuda()
    with torch.no_grad():
        _, logits, hidden = model.initial_inference_device(obs)
    legal = torch.from_numpy((rng.random((N, A)) < 0.7).astype(np.int32)).cuda()
    legal[:, 0] = 1
    noise = torch.from_numpy(rng.dirichlet([0.3] * A, N).astype(np.float32)).cuda()
    return model, logits, hidden, legal, noise


def test_small_search_with_row_executor_selects_the_same_actions():
    """A whole search (eager, capture, replay) with executor='rows' against the same search on the library chain: same
    visit totals, >= 0.99 of the root actions identical (the trees are bit-exact functions of the network outputs,
    which differ in the last fp16 bits), root values within 1e-2."""
    from hanabizero_b200 import _lib, cytree
    from hanabizero_b200.mcts import MCTS
    N, S = 1024, Cfg.num_simulations
    model, logits, hidden, legal, noise = _roots_inputs(N, 4)
    stats = {}
    for ex in ("library", "rows"):
        mcts = MCTS(Cfg)
        before = _lib.gemm_launch_count()
        for _ in range(3):
            roots = cytree.Roots(N, A, S)
            roots.prepare(0.25, noise, torch.zeros(N, device="cuda"), logits.float(), legal)
            mcts.run_multi(roots, model, hidden, executor=ex)
        assert all(ws.chain._use_rows == (ex == "rows") for ws in mcts._ws.values())
        assert ex == "library" or _lib.gemm_launch_count() == before, "the row executor must not run library GEMMs"
        v, val = roots.get_stats_tensors()
        stats[ex] = (v.clone(), val.clone())
    (v0, val0), (v1, val1) = stats["library"], stats["rows"]
    assert int(v1.sum()) == N * (S - 1) and torch.equal(v0.sum(1), v1.sum(1))
    agree = (v0.argmax(1) == v1.argmax(1)).float().mean().item()
    assert agree >= 0.99, agree
    assert (val0 - val1).abs().max().item() < 1e-2


def test_small_search_pipeline_runs_rows_and_equals_serial_searches():
    """SearchPipeline over a Hanabi-Small model (executor 'auto', 3 searches of 2048 trees in flight = 48 row blocks)
    runs the row executor, and every search equals a stand-alone run_multi with the pipeline's own settings, bit for
    bit.  The same model with 3 x 256 trees in flight stays on the library chain (network_executor_for)."""
    from hanabizero_b200 import cytree
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    N, S, depth = 2048, Cfg.num_simulations, 3
    model, logits, hidden, legal, noise = _roots_inputs(N, 7)
    assert SearchPipeline(MCTS(Cfg), model, 256, A, depth=depth).executor == "library"
    pipe = SearchPipeline(MCTS(Cfg), model, N, A, depth=depth)
    assert pipe.executor == "rows"
    rng = np.random.default_rng(11)
    jobs = []
    for k in range(3 * depth):
        jobs.append(dict(noise=torch.from_numpy(rng.dirichlet([0.3] * A, N).astype(np.float32)).cuda(),
                         reward=torch.zeros(N, device="cuda"), logits=(logits.float() + 0.1 * k).contiguous(),
                         legal=legal.clone(), hidden=(hidden * (1.0 + 0.01 * k)).contiguous(),
                         visits=torch.empty(N, A, dtype=torch.int32, device="cuda"), values=torch.empty(N, device="cuda")))
    for j in jobs:
        pipe.submit(0.25, j["noise"], j["reward"], j["logits"], j["legal"], j["hidden"], j["visits"], j["values"])
    pipe.drain()
    torch.cuda.synchronize()
    chains = [ws.chain for ws in pipe.mcts._ws.values()]
    assert len(chains) == depth and all(c._use_rows for c in chains)
    ref = MCTS(Cfg)
    for j in jobs:
        roots = cytree.Roots(N, A, S)
        roots.prepare(0.25, j["noise"], j["reward"], j["logits"], j["legal"])
        ref.run_multi(roots, model, j["hidden"], gemm_sm_target=pipe.gemm_sm_target, stage_limit=pipe.stage_limit,
                      executor=pipe.executor)
        v, val = roots.get_stats_tensors()
        assert torch.equal(v, j["visits"]) and torch.equal(val, j["values"])
        assert int(j["visits"].sum()) == N * (S - 1)


def test_small_selfplay_pool_runs_rows_and_equals_its_engines_stepped_alone():
    """A SelfPlayPool of Hanabi-Small engines (fp16 network, 3 x 2048 games = 48 row blocks in flight) runs the row
    executor, and every engine plays exactly the moves it plays when it is stepped alone with the same settings."""
    from hanabizero_b200.mcts import SearchConfig, gemm_sm_target_for
    from hanabizero_b200.model import MuZeroNet
    from hanabizero_b200.selfplay import SelfPlayEngine, SelfPlayPool
    dev = torch.device("cuda")
    torch.manual_seed(0)
    N, S, E, moves = 2048, 10, 3, 5
    model = MuZeroNet(193 * 4, A).randomize_heads().to(dev).eval()
    cfg = SearchConfig(num_simulations=S, amp_type="torch_amp")
    make = lambda e: SelfPlayEngine(N, "Hanabi-Small", model, cfg, seeds=np.arange(N) + 1000 * e, noise_seed=5,
                                    game_offset=e * N, device=dev)
    alone = []
    for e in range(E):
        eng = make(e)
        eng.gemm_sm_target = gemm_sm_target_for(N, E, dev)
        eng.executor = "rows"
        eng.reset()
        alone.append([{k: v.clone() for k, v in eng.step(deterministic=True).items()} for _ in range(moves)])
    torch.cuda.synchronize()
    engines = [make(e) for e in range(E)]
    pool = SelfPlayPool(engines)
    pool.reset()
    together = []
    for _ in range(moves):
        outs = pool.step(deterministic=True)
        pool.synchronize()
        together.append([{k: v.clone() for k, v in out.items()} for out in outs])
    for eng in engines:
        assert eng.executor == "rows"
        assert all(ws.chain._use_rows for ws in eng.mcts._ws.values() if ws.chain is not None)
        assert any(ws.chain is not None for ws in eng.mcts._ws.values())
    for m in range(moves):
        for e in range(E):
            for k in ("action", "reward", "done", "score", "visits", "root_value"):
                assert torch.equal(together[m][e][k], alone[e][m][k]), (m, e, k)
