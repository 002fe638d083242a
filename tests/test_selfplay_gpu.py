"""GPU: the "next" rows (SURVEY §8f N1/N2) — device select_action, frame stack, and the device-resident
self-play step that chains env + network + search without a host hop."""
import numpy as np
import pytest
import torch

from helpers import ref_select_action

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("temperature", [1.0, 0.5, 0.25])
@pytest.mark.parametrize("deterministic", [True, False])
def test_select_action_matches_reference_rule(temperature, deterministic):
    from hanabizero_b200.selfplay import select_action_batch
    rng = np.random.default_rng(3)
    N, A = 512, 20
    visits = rng.integers(0, 50, (N, A)).astype(np.int32)
    visits[rng.random((N, A)) < 0.5] = 0
    visits[np.arange(N), rng.integers(0, A, N)] += 1
    legal = (rng.random((N, A)) < 0.7).astype(np.float32)
    legal[np.arange(N), visits.argmax(1)] = 1.0
    u = rng.random(N)
    v_dev = torch.from_numpy(visits.copy()).cuda()
    act, ent = select_action_batch(v_dev, torch.from_numpy(legal).cuda(), temperature, deterministic, u)
    act, ent, v_after = act.cpu().numpy(), ent.cpu().numpy(), v_dev.cpu().numpy()
    for i in range(N):
        a, e, vc = ref_select_action(visits[i], temperature, deterministic, legal[i], u[i])
        assert act[i] == a, (i, act[i], a)
        assert abs(ent[i] - e) <= 1e-5 * max(1.0, abs(e))        # fp64 on both sides, float32 output
        assert (v_after[i] == np.asarray(vc)).all()               # illegal counts zeroed in place


def test_select_action_scalar_dropin():
    from hanabizero_b200.selfplay import select_action
    counts = [0, 3, 40, 5, 1]
    a, e = select_action(counts, temperature=1, deterministic=True, legal_actions=[1, 1, 0, 1, 1])
    assert a == 3 and counts[2] == 0 and e > 0


def test_stack_push_matches_torch():
    from hanabizero_b200 import _lib
    lib = _lib.load()
    N, S, D = 37, 4, 785
    stack = torch.rand(N, S, D, device="cuda")
    obs = torch.rand(N, D + 3, device="cuda")
    done = (torch.rand(N, device="cuda") < 0.3).to(torch.uint8)
    want = torch.cat((stack[:, 1:], obs[:, None, :D]), dim=1)
    want[done.bool()] = obs[done.bool()][:, None, :D].expand(-1, S, -1)
    _lib.check(lib.hz_stack_push(torch.cuda.current_stream().cuda_stream, stack.data_ptr(), obs.data_ptr(), obs.stride(0),
                                 done.data_ptr(), N, S, D))
    assert torch.equal(stack, want)


@pytest.mark.parametrize("mdp", ["global", "local"])
def test_selfplay_engine_steps_on_device(mdp):
    from hanabizero_b200.mcts import SearchConfig
    from hanabizero_b200.model import MuZeroNetFull
    from hanabizero_b200.selfplay import SelfPlayEngine
    N, S, stack = 128, 12, 4
    torch.manual_seed(0)
    dim = 785 if mdp == "global" else 660
    model = MuZeroNetFull(dim * stack, 20).randomize_heads().cuda().eval()
    eng = SelfPlayEngine(N, "Hanabi-Full", model, SearchConfig(num_simulations=S), seeds=np.arange(N), mdp=mdp, stack=stack)
    obs, legal = eng.reset()
    assert obs.shape == (N, dim * stack)
    assert eng.iplan is not None                                  # ring of bytes + folded root inference
    fr = lambda: eng.frames_tensor().view(N, stack, dim)          # frame order: oldest first (core/game.py:169-174)
    assert torch.equal(fr()[:, 0], fr()[:, -1])                   # first frame replicated
    total_done = 0
    for t in range(8):
        legal_before = eng.legal.clone()
        prev_last = fr()[:, -1].clone()
        out = eng.step(temperature=1.0, deterministic=(t % 2 == 0))
        a = out["action"].long()
        assert (legal_before.gather(1, a[:, None]) == 1).all()    # only legal moves are played
        assert (out["visits"].sum(1) == S - 1).all()
        d = out["done"].bool()
        total_done += int(d.sum())
        # frame stack: shifted for running games, refilled for restarted ones
        assert torch.equal(fr()[~d][:, -2], prev_last[~d])
        if d.any():
            assert torch.equal(fr()[d][:, 0], fr()[d][:, -1]) and torch.equal(fr()[d][:, 1], fr()[d][:, 2])
        ref_obs = eng.env.observe()[0 if mdp == "global" else 1]
        assert torch.equal(fr()[:, -1], ref_obs)
    eng.env.check()


def test_evaluate_equals_a_reference_style_host_loop():
    """evaluate() (core/test.py:44-126 on the device) against the same loop written the reference's way: scalar
    HanabiEnv objects behind HanabiControlWrapper, list-based cytree calls, the scalar select_action."""
    from hanabizero_b200 import cytree
    from hanabizero_b200.env_wrapper import HanabiControlWrapper
    from hanabizero_b200.hanabi_env import HanabiEnv
    from hanabizero_b200.mcts import MCTS, SearchConfig
    from hanabizero_b200.model import MuZeroNet
    from hanabizero_b200.selfplay import evaluate, select_action
    N, S, stack, A = 6, 8, 4, 11
    torch.manual_seed(0)
    model = MuZeroNet(193 * stack, A).randomize_heads().cuda().eval()
    cfg = SearchConfig(num_simulations=S)
    seeds = [3, 4, 5, 6, 7, 8]
    scores, moves = evaluate(model, cfg, N, "Hanabi-Small", seeds=seeds, mdp="global", stack=stack)

    envs = [HanabiControlWrapper(HanabiEnv({"hanabi_name": "Hanabi-Small", "seed": s}), 0.999, mdp="global") for s in seeds]
    windows, legals = [], []
    for env in envs:
        o, la = env.reset()
        windows.append([o] * stack)
        legals.append(la)
    dones = np.zeros(N, bool)
    ref_scores, ref_moves = [0] * N, [0] * N
    while not dones.all():
        stack_obs = torch.from_numpy(np.array(windows)).cuda().reshape(N, -1)
        out = model.initial_inference(stack_obs.float())
        roots = cytree.Roots(N, A, S)
        roots.prepare_no_noise(out.reward, out.policy_logits.tolist(), legals)
        MCTS(cfg).run_multi(roots, model, out.hidden_state)
        dist = roots.get_distributions()
        for i in range(N):
            if dones[i]:
                continue
            action, _ = select_action(dist[i], temperature=1, deterministic=True, legal_actions=legals[i])
            o, r, d, info, la = envs[i].step(int(action))
            windows[i] = windows[i][1:] + [o]
            legals[i] = la
            dones[i] = bool(d)
            ref_moves[i] += 1
            if dones[i]:
                ref_scores[i] = info.item()["score"]
    assert scores == ref_scores and moves == ref_moves
    assert all(m >= 1 for m in moves)


def test_selfplay_engine_noise_is_reproducible_on_the_host():
    """SelfPlayEngine draws move m's root noise from stream (noise_seed, m, game): regenerating it on the host and
    searching the same roots through the generic calls gives the engine's visit counts."""
    from hanabizero_b200 import cytree
    from hanabizero_b200.mcts import MCTS, SearchConfig
    from hanabizero_b200.model import MuZeroNetFull
    from hanabizero_b200.selfplay import SelfPlayEngine, dirichlet_noise_host
    dev = torch.device("cuda")
    torch.manual_seed(0)
    N, A, S = 32, 20, 12
    model = MuZeroNetFull(785 * 4, A).randomize_heads().to(dev).eval()
    cfg = SearchConfig(num_simulations=S)
    eng = SelfPlayEngine(N, "Hanabi-Full", model, cfg, seeds=np.arange(N), noise_seed=77, game_offset=100, device=dev)
    frames, legal = eng.reset()
    eng.step()                                    # move 0
    frames, legal = eng.frames_tensor().clone(), eng.legal.clone()
    out = eng.step(deterministic=True)            # move 1: its noise is stream (77, 1, 100 + i)
    noise = dirichlet_noise_host(N, A, cfg.root_dirichlet_alpha, seed=77, step=1, root_offset=100)
    with torch.no_grad():
        _, logits, hidden = model.initial_inference_device(frames)
    roots = cytree.Roots(N, A, S, device=dev)
    roots.prepare(cfg.root_exploration_fraction, noise, np.zeros(N, np.float32), logits.float(), legal.int())
    MCTS(cfg).run_multi(roots, model, hidden)
    want = roots.get_distributions_tensor() * (legal > 0).int()     # select_action zeroes the counts of illegal moves
    assert torch.equal(want, out["visits"])


@pytest.mark.parametrize("small", [False, True])
def test_initial_plan_matches_the_module(small):
    """InitialPlan (BN folded, 10 / 5 cuBLASLt GEMMs, frames at a 16-aligned stride) computes initial_inference:
    float32 plan vs the float32 module within 1e-4, the float16 plan within fp16 rounding."""
    from hanabizero_b200 import _lib
    from hanabizero_b200.model import MuZeroNet, MuZeroNetFull
    dev = torch.device("cuda")
    torch.manual_seed(1)
    D, S, A, n = (193, 4, 11, 77) if small else (785, 4, 20, 300)
    model = (MuZeroNet if small else MuZeroNetFull)(D * S, A).randomize_heads().to(dev)
    model.train()
    with torch.no_grad():                      # non-trivial BatchNorm statistics
        for _ in range(3):
            model.initial_inference((torch.rand(64, D * S, device=dev) < 0.2).float())
    model.eval()
    frames = (torch.rand(n, S, D, device=dev) < 0.2).to(torch.uint8)
    lib = _lib.load()
    with torch.no_grad():
        value, logits, state = model.initial_inference_device(frames.float().view(n, -1))
    for dtype, tol in ((torch.float32, 2e-4), (torch.float16, 3e-2)):
        plan = model.initial_plan(dtype, D, S)
        Dp = plan.frame_stride
        ring = torch.zeros(n, S, Dp, dtype=torch.uint8, device=dev)
        head = 2
        for j in range(S):                     # logical frame j lives in ring slot (head + j) % S
            ring[:, (head + j) % S, :D] = frames[:, j]
        b = plan.bound(n)
        _lib.check(lib.hz_ring_gather(torch.cuda.current_stream().cuda_stream, ring.data_ptr(), head, b.x.data_ptr(),
                                      b.x.stride(0), Dp, n, S, Dp, b.x.element_size()))
        want_x = torch.zeros(n, S, Dp, device=dev)
        want_x[:, :, :D] = frames.float()
        assert torch.equal(b.x.float().view(n, S, Dp), want_x)
        v, lg, st = plan.run(n, decode_value=True)
        torch.testing.assert_close(st.float(), state.float(), rtol=tol, atol=tol)
        torch.testing.assert_close(lg, logits, rtol=tol, atol=tol)
        torch.testing.assert_close(v, value, rtol=10 * tol, atol=10 * tol)


def test_selfplay_pool_equals_its_engines_stepped_alone():
    """SelfPlayPool steps several engines on their own streams (their move chains interleave on the GPU); every engine
    must play exactly the moves it plays when it is stepped alone: same actions, rewards, visit counts, scores."""
    from hanabizero_b200.mcts import SearchConfig
    from hanabizero_b200.model import MuZeroNetFull
    from hanabizero_b200.selfplay import SelfPlayEngine, SelfPlayPool
    dev = torch.device("cuda")
    torch.manual_seed(0)
    N, A, S, E, moves = 48, 20, 10, 3, 5
    model = MuZeroNetFull(785 * 4, A).randomize_heads().to(dev).eval()
    cfg = SearchConfig(num_simulations=S, amp_type="torch_amp")
    make = lambda e: SelfPlayEngine(N, "Hanabi-Full", model, cfg, seeds=np.arange(N) + 1000 * e, noise_seed=5,
                                    game_offset=e * N, device=dev)
    from hanabizero_b200.mcts import gemm_sm_target_for
    alone = []
    for e in range(E):
        eng = make(e)
        eng.gemm_sm_target = gemm_sm_target_for(N, E, dev)     # the pool's choice of network kernels => same roundings
        eng.executor = "rows"                                  # (engines in a pool run the row-block resident executor)
        eng.reset()
        alone.append([{k: v.clone() for k, v in eng.step(deterministic=True).items()} for _ in range(moves)])
    torch.cuda.synchronize()
    pool = SelfPlayPool([make(e) for e in range(E)])
    pool.reset()
    together = []
    for _ in range(moves):
        outs = pool.step(deterministic=True)     # arg-max moves: sampled ones draw from torch's global generator
        pool.synchronize()            # the result tensors live on the engines' streams: read them once those are done
        together.append([{k: v.clone() for k, v in out.items()} for out in outs])
    for m in range(moves):
        outs = together[m]
        for e in range(E):
            for k in ("action", "reward", "done", "score", "visits", "root_value"):
                assert torch.equal(outs[e][k], alone[e][m][k]), (m, e, k)
