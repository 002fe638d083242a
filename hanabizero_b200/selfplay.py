"""Device-resident self-play step — the "next" rows of the scope table (SURVEY.md §8f N1, N2) that sit
between the two halves of the hot path in the reference's actor loop
(/root/reference/core/selfplay_worker.py:258-300):

    stack_obs -> initial_inference -> Roots.prepare(noise) -> MCTS.run_multi -> select_action -> env.step

`select_action` is the drop-in for core/utils.py:280-295; `SelfPlayEngine` chains everything for N games
without a host hop: the frame stack (core/game.py:169-174) lives in HBM, the env kernel writes each new
observation straight into it, actions go from the sampler kernel into the env kernel.
"""
import numpy as np
import torch

from . import _lib, cytree
from ._lib import check, ptr
from .hanabi_env import HanabiVecEnv
from .mcts import MCTS


def dirichlet_noise(num, actions, alpha, device, seed=0, step=0, root_offset=0, legal=None):
    """np.random.dirichlet([alpha] * A) per root (selfplay_worker.py:279, reanalyze_worker.py:343), drawn on the
    device from counter-based streams keyed by (seed, step, root_offset + root, action): float32 CUDA [num, actions].
    `legal` (float [num, actions]) zeroes, after normalisation, the entries whose mask value == 0 (-0 included); any
    other value, 0.5 or NaN included, leaves the entry as drawn.  alpha must lie in [1e-300, 1e300].
    `dirichlet_noise_host` returns the same numbers, bit for bit, without a GPU."""
    lib = _lib.load()
    dev = torch.device(device)
    out = torch.empty(num, actions, dtype=torch.float32, device=dev)
    lg = None if legal is None else legal.to(device=dev, dtype=torch.float32).contiguous()
    check(lib.hz_dirichlet_noise(torch.cuda.current_stream(dev).cuda_stream, ptr(out), num, actions, float(alpha),
                                 int(seed) & (2 ** 64 - 1), int(step) & 0xffffffff, int(root_offset), ptr(lg)))
    return out


def dirichlet_noise_host(num, actions, alpha, seed=0, step=0, root_offset=0, legal=None):
    """Host twin of `dirichlet_noise` (hz_host_dirichlet_noise): numpy float32 [num, actions], bit-identical."""
    lib = _lib.load()
    out = np.empty((num, actions), np.float32)
    lg = None if legal is None else np.ascontiguousarray(legal, np.float32)
    check(lib.hz_host_dirichlet_noise(out.ctypes.data, num, actions, float(alpha), int(seed) & (2 ** 64 - 1),
                                      int(step) & 0xffffffff, int(root_offset), None if lg is None else lg.ctypes.data))
    return out


def select_action_batch(visit_counts, legal_actions, temperature=1.0, deterministic=True, uniforms=None):
    """Batched select_action on the device.  visit_counts int32 [N, A] CUDA (illegal entries are zeroed
    in place, as the reference mutates its argument), legal_actions float [N, A].  Non-deterministic
    sampling consumes `uniforms` (float64 [N] in [0, 1); drawn with torch if omitted) through
    numpy.random.choice's inverse-CDF rule.  `temperature` (a number or [N] per row) reaches the kernel as float64, so
    the exponent is Python's 1 / temperature.  Returns (actions int32 [N], entropies float32 [N]); a row left without
    a distribution (no visits on a legal move, or c^(1/T) overflowing) gets action -1 and NaN entropy."""
    n, a = visit_counts.shape
    dev = visit_counts.device
    lib = _lib.load()
    legal = legal_actions.to(device=dev, dtype=torch.float32).contiguous()
    temp = None
    if not (isinstance(temperature, (int, float)) and float(temperature) == 1.0):
        temp = torch.as_tensor(temperature, dtype=torch.float64, device=dev).expand(n).contiguous()
    if deterministic:
        uni = None
    else:
        uni = (torch.rand(n, dtype=torch.float64, device=dev) if uniforms is None
               else torch.as_tensor(uniforms, dtype=torch.float64, device=dev).contiguous())
    actions = torch.empty(n, dtype=torch.int32, device=dev)
    entropy = torch.empty(n, dtype=torch.float32, device=dev)
    check(lib.hz_select_action(torch.cuda.current_stream(dev).cuda_stream, ptr(visit_counts), ptr(legal), ptr(temp),
                               ptr(uni), n, a, ptr(actions), ptr(entropy)))
    return actions, entropy


def select_action(visit_counts, temperature=1, deterministic=True, legal_actions=None):
    """core/utils.py:280-295 for one root: returns (action_pos, count_entropy)."""
    assert legal_actions is not None
    dev = torch.device("cuda", torch.cuda.current_device())
    v = torch.as_tensor(np.asarray(visit_counts), dtype=torch.int32, device=dev).view(1, -1).contiguous()
    lg = torch.as_tensor(np.asarray(legal_actions, dtype=np.float32), device=dev).view(1, -1)
    uni = None if deterministic else np.random.random(1)
    a, e = select_action_batch(v, lg, float(temperature), deterministic, uni)
    zeroed = v[0].cpu().tolist()
    for i, c in enumerate(zeroed):          # the reference mutates the caller's list
        try:
            visit_counts[i] = c
        except TypeError:
            break
    return int(a.item()), float(e.item())


class SelfPlayEngine:
    """N Hanabi games + N trees advanced one move per `step()` entirely on one GPU."""

    def __init__(self, num_games, hanabi_name, model, config, seeds=None, mdp="global", stack=4, device=None,
                 record=False, max_episode_len=128, record_banks=2, noise_seed=0, game_offset=0):
        """record: keep every game's trajectory on the device (hanabizero_b200.trajectory, SURVEY §8f N3);
        finished episodes are fetched with `self.recorder.flush()`.  record=True records on the float frame stack with
        the module's root inference; record="ring" records on the same fast path as an unrecorded engine (byte frame
        ring, InitialPlan root inference, auto-reset in the env launch; the model must have `initial_plan`) with one
        more launch per move.  Both play the moves an unrecorded engine plays.  noise_seed / game_offset key the root
        exploration noise (dirichlet_noise: move m of game i draws stream (noise_seed, m, game_offset + i)), so the
        noise of any move can be regenerated on the host with dirichlet_noise_host."""
        ring = isinstance(record, str)
        if ring and record != "ring":
            raise ValueError(f"record must be False, True or 'ring', got {record!r}")
        if ring and not hasattr(model, "initial_plan"):
            raise ValueError("record='ring' needs a model with initial_plan (the byte frame ring's root inference)")
        self.env = HanabiVecEnv(num_games, hanabi_name, seeds, device=device)
        self.dev, self.n, self.stack, self.mdp = self.env.device, num_games, int(stack), mdp
        self.model, self.config, self.mcts = model, config, MCTS(config)
        self.obs_dim = self.env.global_dim if mdp == "global" else self.env.local_dim
        self.frames = torch.zeros(num_games, self.stack, self.obs_dim, device=self.dev)
        self.legal = torch.zeros(num_games, self.env.num_actions, device=self.dev)
        self.lib = _lib.load()
        self._obs = torch.zeros(num_games, self.obs_dim, device=self.dev)
        self._all_done = torch.ones(num_games, dtype=torch.uint8, device=self.dev)
        # fast path (record=False or "ring"): the frame stack is a ring of 0/1 bytes the env kernel writes into, and the
        # root inference runs as a folded GEMM plan (hanabizero_b200/plan.py InitialPlan) instead of ~70 module kernels
        self.iplan = None
        if (ring or not record) and hasattr(model, "initial_plan"):
            amp = getattr(config, "amp_type", "none") == "torch_amp"
            self.iplan = model.initial_plan(torch.float16 if amp else torch.float32, self.obs_dim, self.stack)
            self.Dp = self.iplan.frame_stride
            self.ring = torch.zeros(num_games, self.stack, self.Dp, dtype=torch.uint8, device=self.dev)
            self.legal8 = torch.zeros(num_games, self.env.num_actions, dtype=torch.uint8, device=self.dev)
            self.head = 0          # ring slot holding the OLDEST frame (the next one to be overwritten)
            if ring:               # terminal rows of the games a move finishes (hz_envs_step_observe_u8_terminal)
                self.term = torch.zeros(num_games, self.Dp, dtype=torch.uint8, device=self.dev)
                self.term_legal = torch.zeros(num_games, self.env.num_actions, dtype=torch.uint8, device=self.dev)
        self.alpha = float(getattr(config, "root_dirichlet_alpha", 0.3))
        self.noise_seed, self.game_offset, self.moves = int(noise_seed), int(game_offset), 0
        self.recorder = None
        self._roots = None
        self.gemm_sm_target = 0      # SelfPlayPool sizes the search's GEMMs for a share of the SMs (mcts.gemm_sm_target_for)
        self.stage_limit = 0         # ... and shrinks the tree step's staging (hz_search_io.stage_limit)
        self.executor = "library"    # ... and runs the network on the row-block resident executor (BoundChain.set_executor)
        if record:
            from .trajectory import TrajectoryRecorder
            self.recorder = TrajectoryRecorder(num_games, self.obs_dim, self.env.num_actions, self.stack,
                                               max_episode_len, device=self.dev, banks=record_banks)

    def _observe_into(self):
        g, l = (self._obs, None) if self.mdp == "global" else (None, self._obs)
        return g, l

    def _observe(self):
        """The current player's observation (the view this engine feeds the network) and legal mask of every game."""
        g, l = self._observe_into()
        check(self.lib.hz_envs_observe(self.env._h, torch.cuda.current_stream(self.dev).cuda_stream, ptr(g),
                                       0 if g is None else g.stride(0), ptr(l), 0 if l is None else l.stride(0),
                                       ptr(self.legal)))

    def _push(self, done):
        check(self.lib.hz_stack_push(torch.cuda.current_stream(self.dev).cuda_stream, ptr(self.frames), ptr(self._obs),
                                     self._obs.stride(0), ptr(done), self.n, self.stack, self.obs_dim))

    def _ring_slot(self, slot):
        """(out_global, out_local) views of ring slot `slot` for the env kernel's byte outputs."""
        row = self.ring[:, slot, :self.obs_dim]
        return (row, None) if self.mdp == "global" else (None, row)

    def _stream(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def reset(self):
        """env.reset() for every game; the first observation fills the whole stack (selfplay_worker.py:137)."""
        self.env.reset_all(observe=False)
        if self.iplan is not None:
            g, l = self._ring_slot(0)
            self.env.observe(out_global=g, out_local=l, out_legal=self.legal8, want_global=g is not None,
                             want_local=l is not None)
            check(self.lib.hz_ring_refill(self._stream(), ptr(self.ring), 0, None, self.n, self.stack, self.Dp))
            self.head = 0
            self.legal.copy_(self.legal8)
            if self.recorder is not None:
                self.recorder.begin(self.ring[:, 0, :self.obs_dim].float(), self.legal)
            return self.frames_tensor(), self.legal
        self._observe()
        self._push(self._all_done)
        if self.recorder is not None:
            self.recorder.begin(self._obs, self.legal)
        return self.frames.view(self.n, -1), self.legal

    def frames_tensor(self):
        """The stacked observation [N, stack * obs_dim] float32, oldest frame first (what the reference feeds
        initial_inference, core/game.py:169-174)."""
        if self.iplan is None:
            return self.frames.view(self.n, -1)
        order = [(self.head + j) % self.stack for j in range(self.stack)]
        return self.ring[:, order, :self.obs_dim].float().reshape(self.n, -1)

    @torch.no_grad()
    def step(self, temperature=1.0, deterministic=False, noise=True):
        """One self-play move for every game.  Returns a dict of CUDA tensors."""
        cfg, n = self.config, self.n
        amp = getattr(cfg, "amp_type", "none") == "torch_amp"
        if self.iplan is not None:
            self.model.eval()
            self.iplan.refresh()
            b = self.iplan.bound(n, owner=self)
            check(self.lib.hz_ring_gather(self._stream(), ptr(self.ring), self.head, ptr(b.x), b.x.stride(0), self.Dp, n,
                                          self.stack, self.Dp, b.x.element_size()))
            _, logits, hidden = self.iplan.run(n, owner=self)
        else:
            with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
                _, logits, hidden = self.model.initial_inference_device(self.frames.view(n, -1))
        # one tree batch per engine, prepared anew every move: its handle (and the search graph captured over it) is
        # never shared with another engine, whose searches may be in flight on another stream (SelfPlayPool)
        if self._roots is None or self._roots.tree_nodes != int(cfg.num_simulations):
            self._roots = cytree.Roots(n, self.env.num_actions, cfg.num_simulations, device=self.dev)
        roots = self._roots
        zeros = torch.zeros(n, device=self.dev)
        legal_i = self.legal.int()
        if noise:   # np.random.dirichlet([alpha] * A) per root (selfplay_worker.py:279), drawn on the device
            nz = dirichlet_noise(n, self.env.num_actions, self.alpha, self.dev, self.noise_seed, self.moves, self.game_offset)
            roots.prepare(cfg.root_exploration_fraction, nz, zeros, logits.float(), legal_i)
        else:
            roots.prepare_no_noise(zeros, logits.float(), legal_i)
        self.mcts.run_multi(roots, self.model, hidden, gemm_sm_target=self.gemm_sm_target, stage_limit=self.stage_limit,
                            executor=self.executor)
        self.moves += 1
        visits, values = roots.get_stats_tensors()
        actions, entropy = select_action_batch(visits, self.legal, temperature, deterministic)
        # env.step for every game; finished games are re-dealt in the same launch and the observation of the
        # current player is written straight into the staging row that feeds the frame stack
        if self.iplan is not None:
            # the new observation replaces the oldest frame in place; finished games get their stack refilled
            slot = self.head
            g, l = self._ring_slot(slot)
            if self.recorder is None:
                _, _, _, reward, done, score = self.env.step_all(actions, auto_reset=True, out_global=g, out_local=l,
                                                                 out_legal=self.legal8, want_global=g is not None,
                                                                 want_local=l is not None)
            else:
                # record="ring": the step also writes finished games' terminal rows (GameHistory.append, game.py:143)
                # before their re-deal, and one launch appends the move and begins the next episodes from the slot
                _, _, _, reward, done, score = self.env.step_all(
                    actions, auto_reset=True, out_global=g, out_local=l, out_legal=self.legal8, want_global=g is not None,
                    want_local=l is not None, out_terminal=self.term[:, :self.obs_dim], out_terminal_legal=self.term_legal)
                self.recorder.record_u8(actions, reward, visits, values, done, self.ring[:, slot], self.legal8, self.term,
                                        self.term_legal)
            check(self.lib.hz_ring_refill(self._stream(), ptr(self.ring), slot, ptr(done), n, self.stack, self.Dp))
            self.head = (slot + 1) % self.stack
            self.legal.copy_(self.legal8)
            return dict(action=actions, reward=reward.clone(), done=done.clone(), score=score.clone(), visits=visits,
                        root_value=values, entropy=entropy)
        g, l = self._observe_into()
        if self.recorder is None:
            _, _, _, reward, done, score = self.env.step_all(actions, auto_reset=True, out_global=g, out_local=l,
                                                             out_legal=self.legal, want_global=g is not None,
                                                             want_local=l is not None)
            self._push(done)
            return dict(action=actions, reward=reward.clone(), done=done.clone(), score=score.clone(), visits=visits,
                        root_value=values, entropy=entropy)
        # recording: the terminal observation belongs to the finished trajectory (GameHistory.append, game.py:143),
        # so the step does not re-deal; finished games are reset by a masked launch after the append
        _, _, _, reward, done, score = self.env.step_all(actions, auto_reset=False, out_global=g, out_local=l,
                                                         out_legal=self.legal, want_global=g is not None,
                                                         want_local=l is not None)
        out = dict(action=actions, reward=reward.clone(), done=done.clone(), score=score.clone(), visits=visits,
                   root_value=values, entropy=entropy, obs=self._obs.clone(), legal=self.legal.clone())
        self.recorder.append(actions, self._obs, self.legal, reward, visits, values, done)
        self.env.reset_all(mask=out["done"], observe=False)
        self._observe()
        self._push(out["done"])
        self.recorder.begin(self._obs, self.legal, mask=out["done"])
        return out


class SelfPlayPool:
    """Several SelfPlayEngines — disjoint game batches, the reference's actors (core/selfplay_worker.py:93-102: each
    DataWorker owns p_mcts_num games) — stepped round-robin, each on its own CUDA stream.  A move is a dependent chain
    of short launches (root inference, search, action pick, env step), so one engine leaves most of the GPU idle; the
    engines' chains interleave and fill one another's gaps.  Nothing here synchronises with the host."""

    def __init__(self, engines):
        self.engines = list(engines)
        if not self.engines:
            raise ValueError("SelfPlayPool needs at least one engine")
        dev = self.engines[0].dev
        self.streams = [torch.cuda.Stream(dev) for _ in self.engines]
        from .mcts import STAGE_LIMIT_IN_FLIGHT, gemm_sm_target_for, network_executor_for
        for eng in self.engines:
            eng.gemm_sm_target = gemm_sm_target_for(eng.n, len(self.engines), dev)
            eng.stage_limit = STAGE_LIMIT_IN_FLIGHT if len(self.engines) > 1 else 0
            eng.executor = network_executor_for(eng.model, eng.n, len(self.engines))
        cur = torch.cuda.current_stream(dev)
        for s in self.streams:
            s.wait_stream(cur)       # engine construction ran on the caller's stream

    def reset(self):
        out = []
        for eng, s in zip(self.engines, self.streams):
            with torch.cuda.stream(s):
                out.append(eng.reset())
        return out

    def step(self, **kw):
        """One move of every engine; returns the engines' result dicts (CUDA tensors, each valid on its engine's
        stream: call synchronize() — or make your stream wait — before reading them elsewhere)."""
        out = []
        for eng, s in zip(self.engines, self.streams):
            with torch.cuda.stream(s):
                out.append(eng.step(**kw))
        return out

    def synchronize(self):
        for s in self.streams:
            s.synchronize()

    def flush(self, store=None):
        """The finished episodes of every recording engine: one list per engine (TrajectoryRecorder.flush; [] for an
        engine that does not record).  Each engine's flush runs on that engine's stream, after its appends.  With
        `store` (trajectory.EpisodeStore) the frames and legal rows go into the store on those streams and the dicts
        carry store ids instead of frames (TrajectoryRecorder.flush(store=...))."""
        out = []
        for eng, s in zip(self.engines, self.streams):
            with torch.cuda.stream(s):
                out.append([] if eng.recorder is None else eng.recorder.flush(store=store))
        return out

    def check(self):
        """TrajectoryRecorder.check of every recording engine, on the engine's stream (synchronises it)."""
        for eng, s in zip(self.engines, self.streams):
            if eng.recorder is not None:
                with torch.cuda.stream(s):
                    eng.recorder.check()


@torch.no_grad()
def evaluate(model, config, num_episodes, hanabi_name="Hanabi-Full", seeds=None, mdp="global", stack=4, max_moves=1000,
             device=None):
    """The evaluation caller of the search (/root/reference/core/test.py:44-126, `test`): `num_episodes` games played to
    the end on the device — noise-free roots (prepare_no_noise), arg-max of the visit counts, finished games stop
    (no re-deal) — one batched search per move.  Returns (final_scores, moves): two int lists, final_scores[i] being
    info['score'] of game i's last step as the reference records it (ep_final_rewards)."""
    env = HanabiVecEnv(num_episodes, hanabi_name, seeds, device=device)
    dev, n, a = env.device, num_episodes, env.num_actions
    lib = _lib.load()
    obs_dim = env.global_dim if mdp == "global" else env.local_dim
    frames = torch.zeros(n, stack, obs_dim, device=dev)
    obs = torch.zeros(n, obs_dim, device=dev)
    legal = torch.zeros(n, a, device=dev)
    g, l = (obs, None) if mdp == "global" else (None, obs)
    st = lambda: torch.cuda.current_stream(dev).cuda_stream
    env.reset_all(observe=False)
    check(lib.hz_envs_observe(env._h, st(), ptr(g), 0 if g is None else g.stride(0), ptr(l),
                              0 if l is None else l.stride(0), ptr(legal)))
    all_games = torch.ones(n, dtype=torch.uint8, device=dev)
    check(lib.hz_stack_push(st(), ptr(frames), ptr(obs), obs.stride(0), ptr(all_games), n, stack, obs_dim))
    alive = torch.ones(n, dtype=torch.uint8, device=dev)
    final = torch.zeros(n, dtype=torch.int32, device=dev)
    moves = torch.zeros(n, dtype=torch.int32, device=dev)
    mcts = MCTS(config)
    model.eval()
    amp = getattr(config, "amp_type", "none") == "torch_amp"
    zeros = torch.zeros(n, device=dev)
    never = torch.zeros(n, dtype=torch.uint8, device=dev)
    for _ in range(max_moves):
        if not bool(alive.any()):
            break
        with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
            _, logits, hidden = model.initial_inference_device(frames.view(n, -1))
        roots = cytree.Roots(n, a, config.num_simulations, device=dev)
        roots.prepare_no_noise(zeros, logits.float(), legal.int())
        mcts.run_multi(roots, model, hidden)
        visits, _ = roots.get_stats_tensors()
        actions, _ = select_action_batch(visits, legal, 1.0, deterministic=True)
        # finished games are not stepped (test.py:99-100) and keep their last observation
        _, _, _, reward, done, score = env.step_all(actions, active=alive, out_global=g, out_local=l, out_legal=legal,
                                                    want_global=g is not None, want_local=l is not None)
        stepped = alive.bool()
        finished = stepped & done.bool()
        final = torch.where(finished, score, final)
        moves += stepped.int()
        check(lib.hz_stack_push(st(), ptr(frames), ptr(obs), obs.stride(0), ptr(never), n, stack, obs_dim))
        alive = (stepped & ~done.bool()).to(torch.uint8)
    env.check()
    return final.cpu().tolist(), moves.cpu().tolist()
