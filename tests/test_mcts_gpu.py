"""GPU: MCTS.run_multi (device-resident loop, CUDA-graph replay, and the compat path around a model that
only speaks the reference's NetworkOutput contract) against the CPU oracle fed the same network outputs."""
import numpy as np
import pytest
import torch

from helpers import nan_to_zero

pytestmark = pytest.mark.gpu

N, A, S = 96, 20, 24


def _setup(amp="none", small=False):
    from hanabizero_b200.hanabi_env import HanabiVecEnv
    from hanabizero_b200.mcts import SearchConfig
    from hanabizero_b200.model import MuZeroNet, MuZeroNetFull
    dev = torch.device("cuda")
    torch.manual_seed(0)
    name, a = ("Hanabi-Small", 11) if small else ("Hanabi-Full", 20)
    env = HanabiVecEnv(N, name, np.arange(N))
    g, _, legal = env.reset_all()
    model = (MuZeroNet if small else MuZeroNetFull)(env.global_dim, a).randomize_heads().to(dev).eval()
    with torch.no_grad():
        _, logits, hidden = model.initial_inference_device(g)
    noise = np.random.default_rng(3).dirichlet([0.3] * a, N).astype(np.float32)
    return dev, model, logits, hidden, legal, noise, SearchConfig(num_simulations=S, amp_type=amp), a


class PlanAsModel:
    """Runs the fused plan through the generic device-resident path (plan.run + hz_trees_backprop_traverse),
    so that its network outputs can be recorded and replayed through the oracle."""

    def __init__(self, plan):
        self.plan = plan

    def eval(self):
        return self

    def recurrent_inference_device(self, h, act):
        state = torch.empty_like(h)
        v, r, lg = self.plan.run(h, act, state)
        return v, r, lg, state


def _record(model):
    """Record (value, reward, logits, hidden_in, action_in, next_state) of every network call of the search."""
    rec = []
    orig = model.recurrent_inference_device

    def wrapped(h, act):
        out = orig(h, act)
        if h.shape[0] == N:   # skip the 2-row dtype probe MCTS makes when it builds its workspace
            rec.append(tuple(o.detach().clone() for o in out[:3]) + (h.detach().clone(), act.detach().clone(), out[3].clone()))
        return out

    model.recurrent_inference_device = wrapped
    return rec, orig


def _oracle_replay(rec, cfg, noise, logits, legal, a):
    from oracle import loader as L
    cpu = L.oracle_tree(N, a, S, cfg.value_delta_max)
    cpu.prepare(0.25, noise, np.zeros(N, np.float32), logits.float().cpu().numpy(), legal.cpu().numpy().astype(np.int32))
    trace = []
    for x, (v, rw, lg, _, _, _) in enumerate(rec, start=1):
        trace.append(cpu.traverse(cfg.pb_c_base, cfg.pb_c_init, cfg.discount))
        cpu.backprop(x, cfg.discount, rw.float().cpu().numpy(), v.float().cpu().numpy(),
                     nan_to_zero(lg.float().cpu().numpy()))
    return cpu, trace


@pytest.mark.parametrize("use_plan", [True, False])
@pytest.mark.parametrize("amp,small", [("none", False), ("torch_amp", False), ("none", True)])
def test_run_multi_matches_oracle_given_same_network_outputs(amp, small, use_plan):
    from hanabizero_b200 import cytree
    from hanabizero_b200.mcts import MCTS
    dev, model, logits, hidden, legal, noise, cfg, a = _setup(amp, small)
    dtype = torch.float16 if amp == "torch_amp" else torch.float32
    net = PlanAsModel(model.recurrent_plan(dtype)) if use_plan else model
    rec, orig = _record(net)
    roots = cytree.Roots(N, a, S)
    roots.prepare(0.25, noise, [0.0] * N, logits, legal)
    MCTS(cfg, use_plan=False).run_multi(roots, net, hidden.to(dtype) if use_plan else hidden, use_graph=False)
    net.recurrent_inference_device = orig
    assert len(rec) == S - 1                               # the last iteration is skipped (core/mcts.py:25-26)
    cpu, trace = _oracle_replay(rec, cfg, noise, logits, legal, a)
    visits, values = roots.get_stats_tensors()
    ov, oval, _ = cpu.stats()
    assert (visits.cpu().numpy() == ov).all()
    np.testing.assert_allclose(values.cpu().numpy(), oval, rtol=1e-5)
    # the batches handed to the network are the parents' hidden states and the last actions
    pool = [(hidden.to(dtype) if use_plan else hidden).to(rec[0][3].dtype)] + [None] * S
    for x, ((v, rw, lg, h, act, nxt), (ix, iy, la)) in enumerate(zip(rec, trace), start=1):
        assert (act.view(-1).cpu().numpy() == la).all()
        want = torch.stack([pool[int(i)][int(j)] for i, j in zip(ix, iy)])
        assert torch.equal(h, want)
        pool[x] = nxt


@pytest.mark.parametrize("amp,small", [("none", False), ("torch_amp", False), ("none", True), ("torch_amp", True)])
def test_fused_search_step_path_equals_generic_path(amp, small):
    """The production path (GEMM chain + hz_trees_search_step decoding raw logits in the tree kernel)
    must give bit-identical trees to the generic path around the same plan, which the test above
    ties to the oracle."""
    from hanabizero_b200 import cytree
    from hanabizero_b200.mcts import MCTS
    dev, model, logits, hidden, legal, noise, cfg, a = _setup(amp, small)
    dtype = torch.float16 if amp == "torch_amp" else torch.float32
    outs = []
    for fused in (True, False):
        roots = cytree.Roots(N, a, S)
        roots.prepare(0.25, noise, [0.0] * N, logits, legal)
        if fused:
            MCTS(cfg, use_plan=True).run_multi(roots, model, hidden, use_graph=False)
        else:
            MCTS(cfg, use_plan=False).run_multi(roots, PlanAsModel(model.recurrent_plan(dtype)), hidden.to(dtype), use_graph=False)
        v, val = roots.get_stats_tensors()
        e = roots.export(S)
        outs.append((v.cpu(), val.cpu(), e["visits"].cpu(), e["value_sum"].cpu(), e["reward"].cpu()))
    for x, y in zip(*outs):
        assert torch.equal(x, y)
    assert (outs[0][0].sum(1) == S - 1).all()


def test_graph_replay_equals_eager_and_is_repeatable():
    from hanabizero_b200 import cytree
    from hanabizero_b200.mcts import MCTS
    dev, model, logits, hidden, legal, noise, cfg, a = _setup()
    mcts = MCTS(cfg)
    outs = []
    for it in range(4):     # 0: eager, 1: capture + replay, 2-3: replay; fresh Roots each time like selfplay
        roots = cytree.Roots(N, a, S)
        nz = noise if it != 3 else np.roll(noise, 1, axis=0)
        roots.prepare(0.25, nz, [0.0] * N, logits, legal)
        mcts.run_multi(roots, model, hidden)
        v, val = roots.get_stats_tensors()
        outs.append((v.cpu().clone(), val.cpu().clone(), roots.export(S)["visits"].cpu().clone()))
        del roots
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][0], outs[2][0])
    assert torch.equal(outs[0][1], outs[1][1]) and torch.equal(outs[0][2], outs[2][2])
    assert not torch.equal(outs[0][0], outs[3][0])         # different noise -> the replay really re-ran the search
    assert (outs[3][0].sum(1) == S - 1).all()


def test_compat_path_with_reference_style_model():
    """A model exposing only recurrent_inference -> NetworkOutput of numpy arrays (core/model.py:74-84)."""
    from hanabizero_b200 import cytree
    from hanabizero_b200.mcts import MCTS
    from hanabizero_b200.model import NetworkOutput
    dev, model, logits, hidden, legal, noise, cfg, a = _setup()

    class RefStyle:
        def __init__(self, m):
            self.m = m

        def eval(self):
            return self

        def recurrent_inference(self, h, act):
            v, r, lg, st = self.m.recurrent_inference_device(h, act)
            return NetworkOutput(v.view(-1, 1).cpu().numpy(), r.view(-1, 1).cpu().numpy(), lg.cpu().numpy(), st.cpu().numpy())

    r1, r2 = cytree.Roots(N, a, S), cytree.Roots(N, a, S)
    for r in (r1, r2):
        r.prepare(0.25, noise, [0.0] * N, logits, legal)
    MCTS(cfg).run_multi(r1, RefStyle(model), hidden.cpu().numpy())
    MCTS(cfg, use_plan=False).search(r2, model, hidden, use_graph=False)
    assert r1.get_distributions() == r2.get_distributions()
    np.testing.assert_allclose(r1.get_values(), r2.get_values(), rtol=1e-5)


@pytest.mark.parametrize("small", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_recurrent_plan_matches_module(small, dtype):
    """The folded/fused plan computes the same function as the nn.Module in eval mode (float
    tolerance: BN folding and fp16 storage reorder roundings; stated here, not bit-exact)."""
    from hanabizero_b200.model import MuZeroNet, MuZeroNetFull
    dev = torch.device("cuda")
    torch.manual_seed(1)
    a, inp = (11, 193) if small else (20, 785)
    net = (MuZeroNet if small else MuZeroNetFull)(inp, a).randomize_heads(std=0.05).to(dev)
    for m in net.modules():      # non-trivial BN statistics
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.normal_(0, 0.2); m.running_var.uniform_(0.5, 1.5)
            m.weight.data.uniform_(0.5, 1.5); m.bias.data.normal_(0, 0.2)
    net.eval()
    n = 257
    hidden = torch.rand(n, 512, device=dev)
    act = torch.randint(0, a, (n, 1), device=dev)
    with torch.no_grad():
        v0, r0, l0, s0 = net.recurrent_inference_device(hidden, act)
    plan = net.recurrent_plan(dtype)
    out_state = torch.empty(n, 512, device=dev, dtype=dtype)
    v1, r1, l1 = plan.run(hidden.to(dtype), act, out_state)
    tol = dict(rtol=2e-4, atol=2e-4) if dtype == torch.float32 else dict(rtol=3e-2, atol=3e-2)
    torch.testing.assert_close(out_state.float(), s0, **tol)
    torch.testing.assert_close(l1, l0, **tol)
    torch.testing.assert_close(v1, v0, **tol)
    torch.testing.assert_close(r1, r0, **tol)
    # weight update -> refresh() re-folds in place (same buffers: captured graphs stay valid)
    ptr_before = plan._w["W1"].data_ptr()
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(1.01)
    assert plan.refresh() and plan._w["W1"].data_ptr() == ptr_before and not plan.refresh()
    with torch.no_grad():
        v2, r2, l2, s2 = net.recurrent_inference_device(hidden, act)
    v3, r3, l3 = plan.run(hidden.to(dtype), act, out_state)
    torch.testing.assert_close(l3, l2, **tol)


def test_plan_and_module_paths_select_the_same_actions():
    from hanabizero_b200 import cytree
    from hanabizero_b200.mcts import MCTS
    dev, model, logits, hidden, legal, noise, cfg, a = _setup()
    outs = []
    for use_plan in (True, False):
        roots = cytree.Roots(N, a, S)
        roots.prepare(0.25, noise, [0.0] * N, logits, legal)
        MCTS(cfg, use_plan=use_plan).run_multi(roots, model, hidden, use_graph=False)
        outs.append(roots.get_stats_tensors())
    agree = (outs[0][0].argmax(1) == outs[1][0].argmax(1)).float().mean().item()
    assert agree > 0.9    # same function up to float rounding of the network; the trees see ~1e-6 different inputs


@pytest.mark.parametrize("depth,on_device", [(2, False), (3, False), (3, True)])
def test_search_pipeline_equals_serial_searches(depth, on_device):
    """SearchPipeline (searches of several slots in flight on their own compute streams, inputs and results moved on
    copy streams) must return, for every submitted search, exactly what a stand-alone Roots.prepare + run_multi returns
    for the same inputs — including when the inputs change from search to search, when a slot is reused (eager search,
    graph capture, replays) and when inputs / outputs are device tensors."""
    from hanabizero_b200 import cytree
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    dev, model, logits, hidden, legal, noise, cfg, a = _setup("torch_amp")
    rng = np.random.default_rng(11)
    mcts = MCTS(cfg)
    pipe = SearchPipeline(mcts, model, N, a, depth=depth)
    if on_device:
        pin = lambda t: t.detach().to(dev).contiguous()
        out = lambda *shape, dtype=torch.float32: torch.empty(*shape, dtype=dtype, device=dev)
    else:
        pin = lambda t: t.detach().cpu().contiguous().pin_memory()
        out = lambda *shape, dtype=torch.float32: torch.empty(*shape, dtype=dtype).pin_memory()
    jobs = []
    for k in range(4 * depth):
        nz = torch.from_numpy(rng.dirichlet([0.3] * a, N).astype(np.float32))
        lg = logits.float().cpu() + 0.1 * k
        hd = hidden.cpu() * (1.0 + 0.01 * k)
        jobs.append(dict(noise=pin(nz) if k % 3 else None, reward=pin(torch.zeros(N)), logits=pin(lg), legal=pin(legal.int()),
                         hidden=pin(hd), visits=out(N, a, dtype=torch.int32), values=out(N)))
    tickets = [pipe.submit(0.25, j["noise"], j["reward"], j["logits"], j["legal"], j["hidden"], j["visits"], j["values"])
               for j in jobs]
    pipe.drain()
    torch.cuda.synchronize()
    assert tickets == [k % depth for k in range(4 * depth)]
    ref = MCTS(cfg)
    for j in jobs:
        roots = cytree.Roots(N, a, S)
        if j["noise"] is None:
            roots.prepare_no_noise(j["reward"], j["logits"], j["legal"])
        else:
            roots.prepare(0.25, j["noise"], j["reward"], j["logits"], j["legal"])
        ref.run_multi(roots, model, j["hidden"], gemm_sm_target=pipe.gemm_sm_target,
                      executor=pipe.executor)                      # same network kernels => same roundings
        v, val = roots.get_stats_tensors()
        assert torch.equal(v.cpu(), j["visits"].cpu()) and torch.equal(val.cpu(), j["values"].cpu())
        assert int(j["visits"].sum()) == N * (S - 1)
