"""GPU: self-play recorded on the byte frame ring (SelfPlayEngine(record="ring")) — the env step that also writes the
terminal rows of finished games (hz_envs_step_observe_u8_terminal), the one-launch record kernel (hz_traj_record_u8),
and the engine and pool built on them, each against an independent path.  Every comparison is exact."""
import numpy as np
import pytest
import torch

from helpers import RefGameHistory

pytestmark = pytest.mark.gpu

GAMES = {"Hanabi-Full": dict(dims={"global": 785, "local": 660}, A=20),
         "Hanabi-Small": dict(dims={"global": 193, "local": 173}, A=11)}
SENTINEL = 0xA5


def _same(ep, ref):        # as tests/test_trajectory_gpu.py compares an episode with the GameHistory port
    assert (ep["o"] == ref.obs_history).all() and ep["o"].shape == ref.obs_history.shape
    assert (ep["a"] == ref.actions).all() and (ep["r"] == ref.rewards).all()
    assert ep["vis"].dtype == np.float64 and (ep["vis"] == ref.child_visits).all()
    assert (ep["root"] == ref.root_values).all()
    assert (ep["la"] == ref.legal_actions).all() and ep["la"].shape == ref.legal_actions.shape


# ---- 1. the env step that writes terminal rows ----------------------------------------------------------------------

@pytest.mark.parametrize("N", [1, 37, 4096])
@pytest.mark.parametrize("mdp", ["global", "local"])
@pytest.mark.parametrize("game", list(GAMES))
def test_terminal_step_equals_step_reset_observe(game, mdp, N):
    """Two envs with the same seeds under the same random legal play: one steps with the terminal-row launch, the other
    with auto_reset=0, a masked reset and a second observe.  A third of the steps leave a random set of games out."""
    from hanabizero_b200.hanabi_env import HanabiVecEnv
    dev = torch.device("cuda")
    seeds = np.arange(N) * 3 + 11
    a_env, b_env = (HanabiVecEnv(N, game, seeds, obs_dtype=torch.uint8) for _ in range(2))
    dim, A = GAMES[game]["dims"][mdp], GAMES[game]["A"]
    ld = dim + 5 if N == 37 else (dim + 15) // 16 * 16      # N = 37: rows not 4-byte aligned (the byte store path)
    main = torch.zeros(N, ld, dtype=torch.uint8, device=dev)
    term = torch.empty(N, ld, dtype=torch.uint8, device=dev)
    legal_a = torch.zeros(N, A, dtype=torch.uint8, device=dev)
    term_legal = torch.empty(N, A, dtype=torch.uint8, device=dev)
    step_b = torch.zeros(N, ld, dtype=torch.uint8, device=dev)
    obs_b = torch.zeros(N, ld, dtype=torch.uint8, device=dev)
    step_legal_b = torch.zeros(N, A, dtype=torch.uint8, device=dev)
    legal_b = torch.zeros(N, A, dtype=torch.uint8, device=dev)
    view = lambda t: dict(out_global=t[:, :dim], want_local=False) if mdp == "global" else \
        dict(out_local=t[:, :dim], want_global=False)
    a_env.reset_all(observe=False)
    b_env.reset_all(observe=False)
    a_env.observe(out_legal=legal_a, **view(main))
    b_env.observe(out_legal=legal_b, **view(obs_b))
    assert torch.equal(main, obs_b)
    gen = torch.Generator(device=dev).manual_seed(N)
    steps = 220 if game == "Hanabi-Full" else 120     # a Hanabi-Small episode lasts at most ~30 moves
    finished = torch.zeros(N, dtype=torch.int64, device=dev)
    for t in range(steps):
        actions = torch.multinomial(legal_b.float(), 1, generator=gen).view(-1).int()
        active = None
        if t % 3 == 2:
            active = (torch.rand(N, generator=gen, device=dev) < 0.6).to(torch.uint8)
        term.fill_(SENTINEL)
        term_legal.fill_(SENTINEL)
        a_env.step_all(actions, active=active, auto_reset=True, out_legal=legal_a, out_terminal=term[:, :dim],
                       out_terminal_legal=term_legal, **view(main))
        b_env.step_all(actions, active=active, auto_reset=False, out_legal=step_legal_b, **view(step_b))
        for k in ("reward", "done", "score"):
            assert torch.equal(getattr(a_env, k), getattr(b_env, k)), (t, k)
        fin = b_env.done.bool() if active is None else b_env.done.bool() & active.bool()
        b_env.reset_all(mask=fin.to(torch.uint8), observe=False)
        b_env.observe(out_legal=legal_b, **view(obs_b))
        finished += fin.long()
        # finished games: terminal rows = the step rows of auto_reset=0, main rows = the observation after the reset
        assert torch.equal(term[fin, :dim], step_b[fin, :dim]), t
        assert torch.equal(term_legal[fin], step_legal_b[fin]), t
        assert (term_legal[fin].sum(1) > 0).all()          # no terminal check: the mask is not empty
        assert (term[fin, dim:] == SENTINEL).all()          # nothing past the view's width
        assert torch.equal(main[:, :dim], obs_b[:, :dim]) and torch.equal(legal_a, legal_b), t
        assert torch.equal(main[~fin, :dim], step_b[~fin, :dim]), t
        # unfinished (and skipped) games: their terminal rows are not touched
        assert (term[~fin] == SENTINEL).all() and (term_legal[~fin] == SENTINEL).all(), t
        assert torch.equal(a_env.dump(), b_env.dump()), t
    a_env.check()
    b_env.check()
    assert int(finished.min()) >= 2                         # every game finished several times


def test_terminal_step_argument_rules():
    from hanabizero_b200.hanabi_env import HanabiVecEnv
    env = HanabiVecEnv(4, "Hanabi-Small", np.arange(4), obs_dtype=torch.uint8)
    env.reset_all(observe=False)
    acts = torch.zeros(4, dtype=torch.int32, device="cuda")
    term, tl = torch.zeros(4, 208, dtype=torch.uint8, device="cuda"), torch.zeros(4, 11, dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError):                     # auto_reset is the point of the terminal rows
        env.step_all(acts, auto_reset=False, want_local=False, out_terminal=term, out_terminal_legal=tl)
    with pytest.raises(ValueError):                     # two views: which one would the terminal row be in?
        env.step_all(acts, auto_reset=True, out_terminal=term, out_terminal_legal=tl)
    with pytest.raises(TypeError):                      # byte outputs only
        env.step_all(acts, auto_reset=True, want_local=False, out_global=torch.zeros(4, 193, device="cuda"),
                     out_legal=torch.zeros(4, 11, device="cuda"), out_terminal=term, out_terminal_legal=tl)
    from hanabizero_b200 import _lib
    with pytest.raises(_lib.HzError, match="terminal row stride"):
        env.step_all(acts, auto_reset=True, want_local=False, out_terminal=term[:, :192].contiguous(),
                     out_terminal_legal=tl)


# ---- 2. the record kernel --------------------------------------------------------------------------------------------

def _recorders(N, D, A, stack, max_len, banks):
    from hanabizero_b200.trajectory import TrajectoryRecorder
    return [TrajectoryRecorder(N, D, A, stack, max_len=max_len, banks=banks) for _ in range(2)]


BUFFERS = ("obs", "legal", "action", "reward", "visits", "root_value", "len", "bank", "finished", "overflow")


def _drive(N, D, A, stack, max_len, banks, steps, p_done, flush_every, seed):
    """Random moves through hz_traj_record_u8 (recorder 0) and hz_traj_append + hz_traj_begin(mask=done) fed float
    copies of the same rows (recorder 1); every buffer of the two views must be equal after every move."""
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(seed)
    rec, ref = _recorders(N, D, A, stack, max_len, banks)
    ld_next, ld_term = (D + 15) // 16 * 16 + 16, D + 7
    rows = lambda ld: torch.randint(0, 3, (N, ld), generator=g, device=dev, dtype=torch.uint8)   # 2: any non-zero is 1
    first, first_legal = rows(ld_next), rows(A).contiguous()
    rec.begin(first.float()[:, :D], first_legal.float())
    ref.begin(first.float()[:, :D], first_legal.float())
    overflowed = False
    for t in range(steps):
        nxt, nxt_legal, trm, trm_legal = rows(ld_next), rows(A).contiguous(), rows(ld_term), rows(A).contiguous()
        acts = torch.randint(0, A, (N,), generator=g, device=dev, dtype=torch.int32)
        rew = torch.randint(-1, 3, (N,), generator=g, device=dev, dtype=torch.int32)
        vis = torch.randint(0, 30, (N, A), generator=g, device=dev, dtype=torch.int32)
        root = torch.randn(N, generator=g, device=dev)
        done = (torch.rand(N, generator=g, device=dev) < p_done).to(torch.uint8)
        active = None if t % 4 == 0 else (torch.rand(N, generator=g, device=dev) < 0.8).to(torch.uint8)
        rec.record_u8(acts, rew, vis, root, done, nxt[:, :D], nxt_legal, trm[:, :D], trm_legal, active=active)
        d = done.bool()[:, None]
        app = torch.where(d, trm[:, :D].float(), nxt[:, :D].float())
        app_legal = torch.where(d, trm_legal.float(), nxt_legal.float())
        ref.append(acts, app, app_legal, rew, vis, root, done, active)
        ref.begin(nxt.float()[:, :D], nxt_legal.float(), mask=done)
        for k in BUFFERS:
            assert torch.equal(getattr(rec, k), getattr(ref, k)), (t, k)
        overflowed |= bool(rec.overflow.item())
        if flush_every and t % flush_every == flush_every - 1:
            a, b = rec.flush(), ref.flush()
            assert len(a) == len(b)
            for x, y in zip(a, b):
                assert x["game"] == y["game"] and all(np.array_equal(x[k], y[k]) for k in x if k != "game")
    return overflowed


@pytest.mark.parametrize("stack", [1, 4])
@pytest.mark.parametrize("banks", [2, 3, 4])
@pytest.mark.parametrize("D", [785, 660, 193, 173])
def test_record_kernel_equals_append_then_begin(D, banks, stack):
    A = 20 if D in (785, 660) else 11
    # flushes every banks - 1 moves at most: a game can finish one episode per move
    assert not _drive(37, D, A, stack, max_len=48, banks=banks, steps=40, p_done=0.3, flush_every=banks - 1,
                      seed=D * 10 + banks * 2 + stack)


@pytest.mark.parametrize("cause", ["max_len", "banks"])
def test_record_kernel_overflow_equals_append_then_begin(cause):
    """Both ways a game runs out of room — an episode longer than max_len, every bank holding an unflushed episode —
    leave the same buffers and the same sticky overflow flag as the two-launch sequence.  One game: with several, the
    games that overflow in the same launch race for the flag."""
    if cause == "max_len":
        assert _drive(1, 193, 11, 4, max_len=3, banks=3, steps=30, p_done=0.1, flush_every=0, seed=1)
    else:
        assert _drive(1, 785, 20, 4, max_len=24, banks=2, steps=30, p_done=0.5, flush_every=0, seed=2)


# ---- 3-6. the engine ------------------------------------------------------------------------------------------------

def _model(game, mdp, stack=4):
    from hanabizero_b200.model import MuZeroNet, MuZeroNetFull
    torch.manual_seed(0)
    net = MuZeroNetFull if game == "Hanabi-Full" else MuZeroNet
    return net(GAMES[game]["dims"][mdp] * stack, GAMES[game]["A"]).randomize_heads().cuda().eval()


@pytest.mark.parametrize("amp", ["none", "torch_amp"])
@pytest.mark.parametrize("mdp", ["global", "local"])
@pytest.mark.parametrize("game", list(GAMES))
def test_ring_recording_plays_the_unrecorded_moves(game, mdp, amp):
    from hanabizero_b200.mcts import SearchConfig
    from hanabizero_b200.selfplay import SelfPlayEngine
    N, S, moves = 64, 8, 100
    model = _model(game, mdp)
    cfg = SearchConfig(num_simulations=S, amp_type=amp)
    runs = []
    for record in (False, "ring"):
        eng = SelfPlayEngine(N, game, model, cfg, seeds=np.arange(N) + 3, mdp=mdp, record=record, record_banks=4)
        assert eng.iplan is not None
        torch.manual_seed(7)                  # sampled moves draw their uniforms from torch's generator
        eng.reset()
        runs.append([{k: v.clone() for k, v in eng.step(temperature=1.0, deterministic=False).items()}
                     for _ in range(moves)])
        eng.env.check()
    for m in range(moves):
        assert set(runs[0][m]) == set(runs[1][m])
        for k in ("action", "visits", "root_value", "reward", "done", "score", "entropy"):
            assert torch.equal(runs[0][m][k], runs[1][m][k]), (m, k)
    assert sum(int(r["done"].sum()) for r in runs[1]) > 0


@pytest.mark.parametrize("game,mdp", [("Hanabi-Full", "global"), ("Hanabi-Small", "local"), ("Hanabi-Small", "global")])
def test_ring_episodes_equal_an_independent_replay(game, mdp):
    """The engine's actions replayed through a float HanabiVecEnv without auto-reset (masked resets after the step),
    fed with the engine's visits and root values into the GameHistory port; every flushed episode — terminal
    observation included — must equal the port's.  Flushes at irregular moves and a reset() halfway."""
    from hanabizero_b200.hanabi_env import HanabiVecEnv
    from hanabizero_b200.mcts import SearchConfig
    from hanabizero_b200.selfplay import SelfPlayEngine
    N, S, stack, moves = 48, 6, 4, 90
    seeds = np.arange(N) + 5
    eng = SelfPlayEngine(N, game, _model(game, mdp, stack), SearchConfig(num_simulations=S), seeds=seeds, mdp=mdp,
                         stack=stack, record="ring", max_episode_len=128, record_banks=4)
    rep = HanabiVecEnv(N, game, seeds)
    view = lambda g, l: (g if mdp == "global" else l).cpu().numpy()
    refs = [RefGameHistory(stack) for _ in range(N)]
    want, got = [[] for _ in range(N)], [[] for _ in range(N)]

    def begin_all():
        eng.reset()
        g, l, legal = rep.reset_all()
        o, la = view(g, l), legal.cpu().numpy().astype(np.float64)
        assert (eng.frames_tensor().view(N, stack, -1)[:, -1].cpu().numpy() == o).all()
        for i in range(N):
            refs[i] = RefGameHistory(stack)
            refs[i].init([o[i]] * stack, la[i])

    def collect():
        for ep in eng.recorder.flush():
            got[ep["game"]].append(ep)

    begin_all()
    flush_at = {1, 3, 4, 7, 9, 10, 12, 13, 16, 19}              # gaps of 1..3 moves: four banks never fill
    flush_at |= {m + 20 * k for m in flush_at for k in range(1, 5)}
    for t in range(moves):
        if t == moves // 2:                                      # partial episodes are dropped, finished ones kept
            begin_all()
        out = eng.step(temperature=1.0, deterministic=False)
        h = {k: v.cpu().numpy() for k, v in out.items()}
        g, l, legal, reward, done, _ = rep.step_all(out["action"], auto_reset=False)
        o, la = view(g, l), legal.cpu().numpy().astype(np.float64)
        assert (reward.cpu().numpy() == h["reward"]).all() and (done.cpu().numpy() == h["done"]).all()
        for i in range(N):
            refs[i].store_search_stats(h["visits"][i].tolist(), float(h["root_value"][i]))
            refs[i].append(int(h["action"][i]), o[i], int(h["reward"][i]), la[i])
        if h["done"].any():
            g, l, legal = rep.reset_all(mask=done.clone())
            o, la = view(g, l), legal.cpu().numpy().astype(np.float64)
            for i in np.flatnonzero(h["done"]):
                refs[i].game_over(); refs[i].put()
                want[i].append(refs[i])
                refs[i] = RefGameHistory(stack)
                refs[i].init([o[i]] * stack, la[i])
        if t in flush_at:
            collect()
    collect()
    eng.env.check()
    rep.check()
    assert sum(len(w) for w in want) >= N
    for i in range(N):
        assert len(got[i]) == len(want[i]), i
        for ep, ref in zip(got[i], want[i]):
            _same(ep, ref)
            assert len(ep["a"]) + stack == len(ep["o"]) and len(ep["la"]) == len(ep["a"]) + 1


@pytest.mark.parametrize("cause", ["max_len", "banks"])
def test_ring_recording_reports_overflow(cause):
    from hanabizero_b200.mcts import SearchConfig
    from hanabizero_b200.selfplay import SelfPlayEngine
    from hanabizero_b200.trajectory import TrajectoryOverflow
    N = 32
    if cause == "max_len":      # a Hanabi-Full episode lasts at least three moves
        eng = SelfPlayEngine(N, "Hanabi-Full", _model("Hanabi-Full", "global"), SearchConfig(num_simulations=4),
                             record="ring", max_episode_len=2)
    else:                       # Hanabi-Small episodes are short: two banks fill without a flush
        eng = SelfPlayEngine(N, "Hanabi-Small", _model("Hanabi-Small", "global"), SearchConfig(num_simulations=4),
                             record="ring", record_banks=2)
    eng.reset()
    for _ in range(2 if cause == "max_len" else 1):     # not yet: two moves fill max_len, one move finishes one bank
        eng.step()
    eng.recorder.check()
    for _ in range(30):
        eng.step()
    with pytest.raises(TrajectoryOverflow):
        eng.recorder.check()


def test_pool_flush_equals_engines_flushed_alone():
    """SelfPlayPool of recording engines, flushed with pool.flush() (each engine's flush on its own stream): the same
    episodes, bit for bit, as every engine stepped and flushed alone."""
    from hanabizero_b200.mcts import STAGE_LIMIT_IN_FLIGHT, SearchConfig, gemm_sm_target_for, network_executor_for
    from hanabizero_b200.selfplay import SelfPlayEngine, SelfPlayPool
    dev = torch.device("cuda")
    N, S, E, moves = 48, 8, 3, 24
    model = _model("Hanabi-Small", "global")
    cfg = SearchConfig(num_simulations=S, amp_type="torch_amp")
    make = lambda e: SelfPlayEngine(N, "Hanabi-Small", model, cfg, seeds=np.arange(N) + 1000 * e, noise_seed=5,
                                    game_offset=e * N, device=dev, record="ring", record_banks=4)
    flush = lambda m: m % 3 == 2
    alone = []
    for e in range(E):
        eng = make(e)
        eng.gemm_sm_target = gemm_sm_target_for(N, E, dev)     # the pool's choices of network kernels => same roundings
        eng.stage_limit = STAGE_LIMIT_IN_FLIGHT
        eng.executor = network_executor_for(model, N, E)
        eng.reset()
        eps = []
        for m in range(moves):
            eng.step(deterministic=True)
            if flush(m):
                eps += eng.recorder.flush()
        eps += eng.recorder.flush()
        alone.append(eps)
    pool = SelfPlayPool([make(e) for e in range(E)])
    pool.reset()
    together = [[] for _ in range(E)]
    for m in range(moves):
        pool.step(deterministic=True)
        if flush(m):
            for e, eps in enumerate(pool.flush()):
                together[e] += eps
    pool.check()
    for e, eps in enumerate(pool.flush()):
        together[e] += eps
    assert sum(len(a) for a in alone) >= N
    for e in range(E):
        assert len(together[e]) == len(alone[e]), e
        for x, y in zip(together[e], alone[e]):
            assert x["game"] == y["game"] and all(np.array_equal(x[k], y[k]) for k in x if k != "game"), e
