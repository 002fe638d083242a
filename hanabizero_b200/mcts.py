"""Search driver: drop-in for the reference's core/mcts.py (MCTS.run_multi, :7-57; `search` is
the upstream-EfficientZero alias BASELINE.json uses).

The reference loop crosses the host twice per simulation (Python-list marshalling into C++, a
Python gather of hidden states, H2D of the batch, D2H + .tolist() of the network output).  Here a
simulation is, on the device and on one stream:

    [backprop of sim k-1 + traverse of sim k + gather of the parents' hidden states]  (1 launch)
    -> model.recurrent_inference_device (PyTorch, cuBLAS)  -> next hidden state into pool[k]

and the whole `num_simulations - 1` loop is captured in a CUDA graph after the first search with
a given (tree handle, model, shape), so a search is one graph launch.  Exactly like the reference
the last iteration is skipped (core/mcts.py:25-26): `num_simulations - 1` simulations run.

Models: anything exposing `recurrent_inference_device(hidden, action) -> (value[N], reward[N],
policy_logits[N, A], next_hidden[N, F])` on CUDA (hanabizero_b200.model does) gets the
device-resident path.  A model with only the reference's `recurrent_inference` (numpy or tensor
NetworkOutput) still works through the same kernels, paying that model's own host hops.
"""
import contextlib
import time
import weakref

import numpy as np
import torch

from . import _lib, cytree
from ._lib import check, ptr
from .dist import wave_rows


class SearchConfig:
    """The hot-path constants of BaseMuZeroConfig (core/config.py:105-111) and the Hanabi configs
    (config/hanabi_control/__init__.py:25-28,143-146) for callers without a reference config."""

    def __init__(self, num_simulations=50, discount=0.999, value_delta_max=0.006, pb_c_base=19652,
                 pb_c_init=1.25, amp_type="none", root_dirichlet_alpha=0.3,
                 root_exploration_fraction=0.25):
        if int(num_simulations) < 2:
            # the last simulation is skipped (core/mcts.py:25-26): one simulation leaves the root without visits, and
            # neither a move nor a policy target is defined from zero counts
            raise ValueError(f"num_simulations = {num_simulations}: a search needs at least 2")
        self.num_simulations = num_simulations
        self.discount = discount
        self.value_delta_max = value_delta_max
        self.pb_c_base = pb_c_base
        self.pb_c_init = pb_c_init
        self.amp_type = amp_type
        self.root_dirichlet_alpha = root_dirichlet_alpha
        self.root_exploration_fraction = root_exploration_fraction


class _Workspace:
    """Static device buffers of one (tree handle, model, shape): hidden-state pool [S, N, F], the
    gathered batch handed to the model, the min/max statistics, and the captured graph."""

    def __init__(self, roots, model, sims, feature, dtype):
        n, dev = roots.root_num, roots.device
        self.model_ref = weakref.ref(model)   # id(model) can be recycled: a hit must be for the same live object
        self.chain = None                     # the BoundChain a captured graph points into (kept alive with it)
        self.pool = torch.empty(sims, n, feature, dtype=dtype, device=dev)
        self.hidden = torch.empty(n, feature, dtype=dtype, device=dev)
        self.action64 = torch.zeros(n, 1, dtype=torch.int64, device=dev)
        self.ix = torch.empty(n, dtype=torch.int32, device=dev)
        self.la = torch.empty(n, dtype=torch.int32, device=dev)
        self.minmax = cytree.MinMaxStatsList(n)
        self.minmax.tensor(dev)
        self.graph = None
        self.searches = 0


class MCTS(object):
    max_cached_workspaces = 8

    def __init__(self, config, use_plan=True):
        self.config = config
        self.use_plan = use_plan
        self._ws = {}
        cytree.on_handle_destroyed(self._forget_handle)

    def _forget_handle(self, handle_value):
        """A cached tree batch was destroyed: graphs captured over its buffers must never be replayed."""
        for key in [k for k in self._ws if k[0] == handle_value]:
            del self._ws[key]

    # ---------------------------------------------------------------------------------------------
    def _autocast(self):
        if getattr(self.config, "amp_type", "none") == "torch_amp":  # core/mcts.py:38-40
            return torch.autocast("cuda", dtype=torch.float16)
        return contextlib.nullcontext()

    def _plan(self, model):
        """The model's fused eval-mode plan (hanabizero_b200/plan.py) if it offers one and use_plan is on."""
        if not self.use_plan or not hasattr(model, "recurrent_plan"):
            return None
        amp = getattr(self.config, "amp_type", "none") == "torch_amp"
        return model.recurrent_plan(torch.float16 if amp else torch.float32)

    def pool_dtype(self, model, feature, device):
        """Element type of the hidden-state pool a search of `model` keeps (root hidden states are converted to it)."""
        if self._plan(model) is not None:
            return self._plan(model).dtype
        if hasattr(model, "recurrent_inference_device"):
            with torch.no_grad(), self._autocast():
                probe = model.recurrent_inference_device(
                    torch.zeros(2, feature, device=device), torch.zeros(2, 1, dtype=torch.int64, device=device))
            return probe[3].dtype
        return torch.float32

    def _workspace(self, roots, model, hidden_state_roots, gemm_sm_target=0, stage_limit=0, executor="library"):
        sims = int(self.config.num_simulations)
        key = (roots.handle.value, id(model), sims, getattr(self.config, "amp_type", "none"), self.use_plan,
               int(gemm_sm_target), int(stage_limit), executor)
        ws = self._ws.get(key)
        if ws is not None and ws.model_ref() is not model:
            ws = None   # a different model object that happens to live at a recycled address
        if ws is None:
            feature = int(hidden_state_roots.shape[-1])
            dtype = self.pool_dtype(model, feature, roots.device)
            if len(self._ws) >= self.max_cached_workspaces:
                self._ws.pop(next(iter(self._ws)))
            ws = self._ws[key] = _Workspace(roots, model, sims, feature, dtype)
            ws.gemm_sm_target, ws.stage_limit, ws.executor = int(gemm_sm_target), int(stage_limit), executor
        return ws

    def _simulate(self, roots, model, ws):
        """The device-resident loop; everything is enqueued on the current stream (capturable)."""
        cfg, lib, h = self.config, roots._lib, roots.handle
        sims = int(cfg.num_simulations)
        st = torch.cuda.current_stream(roots.device).cuda_stream
        mm = ws.minmax
        mm.set_delta(cfg.value_delta_max)
        mm.clear()
        mmp = ptr(mm.tensor(roots.device))
        row_bytes = ws.hidden.shape[1] * ws.hidden.element_size()
        base, init, disc, delta = int(cfg.pb_c_base), float(cfg.pb_c_init), float(cfg.discount), float(cfg.value_delta_max)
        if sims < 2:
            return
        check(lib.hz_trees_traverse(h, st, base, init, disc, mmp, delta, ptr(ws.ix), None, ptr(ws.la),
                                    ptr(ws.action64), ptr(ws.pool), ptr(ws.hidden), row_bytes))
        for x in range(1, sims):
            with self._autocast():
                value, reward, logits, state = model.recurrent_inference_device(ws.hidden, ws.action64)
            ws.pool[x].copy_(state)
            value = value.float().contiguous()
            reward = reward.float().contiguous()
            logits = logits.float().contiguous()
            if x < sims - 1:
                check(lib.hz_trees_backprop_traverse(
                    h, st, x, disc, ptr(reward), ptr(value), ptr(logits), 1, mmp, delta, base, init,
                    ptr(ws.ix), None, ptr(ws.la), ptr(ws.action64), ptr(ws.pool), ptr(ws.hidden), row_bytes))
            else:
                check(lib.hz_trees_backprop(h, st, x, disc, ptr(reward), ptr(value), ptr(logits), 1, mmp))

    def _simulate_chain(self, roots, plan, ws):
        """Device-resident loop on the fused plan: per simulation one GEMM chain (7 or 5 cuBLASLt
        launches) and ONE tree launch that decodes the raw value/reward logits, expands, back-propagates,
        stores the new hidden state in the pool, traverses and writes the next [hidden ‖ one-hot] batch."""
        cfg, lib, h = self.config, roots._lib, roots.handle
        sims = int(cfg.num_simulations)
        st = torch.cuda.current_stream(roots.device).cuda_stream
        mm = ws.minmax
        mm.set_delta(cfg.value_delta_max)
        mm.clear()
        if sims < 2:
            return
        if ws.chain is None or ws.chain.plan is not plan:
            # the workspace owns its chain (activation buffers + cuBLASLt plan): searches of different tree batches may
            # run on different streams at the same time (SearchPipeline), and a captured graph keeps its buffers alive
            from .plan import BoundChain
            ws.chain = BoundChain(plan, roots.root_num)
            if ws.gemm_sm_target:
                ws.chain.set_sm_target(ws.gemm_sm_target)
            if ws.executor == "rows" and ws.chain.rows_supported():
                ws.chain.set_executor("rows")
        ch = ws.chain
        io = _lib.SearchIO()
        io.value_logits, io.ld_value = ptr(ch.value_logits), ch.value_logits.stride(0)
        io.reward_logits, io.ld_reward = ptr(ch.reward_logits), ch.reward_logits.stride(0)
        io.policy_logits, io.ld_policy = ptr(ch.policy_logits), ch.policy_logits.stride(0)
        io.next_state, io.ld_state = None, 0      # the dynamics GEMM writes pool[x] itself (BoundChain.bind_state)
        io.support, io.support_width, io.support_delta = ptr(plan.support), plan.n_support, plan.net.support_delta
        io.elem_bytes, io.sanitize_nan = ch.x0.element_size(), 1
        io.pool, io.state_cols = ptr(ws.pool), plan.F
        io.out_batch, io.ld_batch, io.onehot_cols = ptr(ch.x0), ch.x0.stride(0), plan.OH
        io.out_ix, io.out_action = ptr(ws.ix), ptr(ws.la)
        io.minmax, io.value_delta_max = ptr(mm.tensor(roots.device)), float(cfg.value_delta_max)
        io.discount, io.pb_c_base, io.pb_c_init = float(cfg.discount), int(cfg.pb_c_base), float(cfg.pb_c_init)
        io.stage_limit = ws.stage_limit
        ref = _lib.C.byref(io)
        check(lib.hz_trees_search_step(h, st, 0, 1, ref))
        for x in range(1, sims):
            ch.bind_state(ws.pool[x])
            ch.run(st)
            check(lib.hz_trees_search_step(h, st, x, 1 if x < sims - 1 else 0, ref))

    def _simulate_compat(self, roots, model, ws):
        """Same kernels around a model that only speaks the reference's NetworkOutput contract."""
        cfg = self.config
        sims = int(cfg.num_simulations)
        mm = ws.minmax
        mm.set_delta(cfg.value_delta_max)
        mm.clear()
        for x in range(1, sims):
            results = cytree.ResultsWrapper(roots.root_num)
            cytree.multi_traverse(roots, cfg.pb_c_base, cfg.pb_c_init, cfg.discount, mm, results,
                                  as_tensor=True, pool=ws.pool, out_hidden=ws.hidden, out_action64=ws.action64)
            with self._autocast():
                out = model.recurrent_inference(ws.hidden.float(), ws.action64)
            dev = roots.device
            ws.pool[x].copy_(cytree.as_device(out.hidden_state, ws.pool.dtype, dev))
            cytree.multi_back_propagate(x, cfg.discount, _flat(out.reward), _flat(out.value),
                                        out.policy_logits, mm, results, sanitize_nan=True)

    # ---------------------------------------------------------------------------------------------
    def run_multi(self, roots, model, hidden_state_roots, use_graph=True, gemm_sm_target=0, stage_limit=0,
                  executor="library"):
        """core/mcts.py:11-57.  roots: cytree.Roots already prepared; hidden_state_roots: [N, F]
        numpy array or tensor (any device).  Mutates `roots` in place and returns None.
        gemm_sm_target > 0 sizes the network's library GEMMs for that many SMs instead of the whole device (for callers
        that keep several searches in flight on different streams: SearchPipeline sets it); stage_limit > 0 likewise
        shrinks the tree step's shared-memory staging so that it shares SMs with other searches' GEMMs
        (hz_search_io.stage_limit).  executor="rows" runs the network as one row-block resident launch per simulation
        (BoundChain.set_executor; fp16 plans of Hanabi-Full and Hanabi-Small, otherwise ignored).  None of them changes any result of the
        tree step; the SM target and the executor change network roundings in the last bits."""
        with torch.no_grad():
            if getattr(model, "training", True):
                model.eval()          # walks every submodule: only when something is still in training mode
            ws = self._workspace(roots, model, hidden_state_roots, gemm_sm_target, stage_limit, executor)
            if self._plan(model) is not None:
                self._plan(model).refresh()   # re-fold weights in place if the module was updated
            ws.pool[0].copy_(cytree.as_device(hidden_state_roots, ws.pool.dtype, roots.device))
            sims = int(self.config.num_simulations)
            plan = self._plan(model)
            if plan is not None:
                simulate = lambda: self._simulate_chain(roots, plan, ws)
            else:
                simulate = lambda: self._simulate(roots, model, ws)
            if plan is None and not hasattr(model, "recurrent_inference_device"):
                self._simulate_compat(roots, model, ws)
            elif not use_graph:
                simulate()
            elif ws.graph is None and ws.searches == 0:
                simulate()  # first search runs eagerly (also warms cuBLAS)
            else:
                if ws.graph is None:
                    torch.cuda.synchronize(roots.device)
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph):
                        simulate()
                    ws.graph = graph
                ws.graph.replay()
                # host-side progress of the handle is not touched by a replay
                check(roots._lib.hz_trees_set_progress(roots.handle, max(sims - 1, 0)))
            ws.searches += 1

    search = run_multi  # upstream EfficientZero name (BASELINE.json north_star)


def _as_tensor(x):
    """A torch tensor of `x` (numpy, lists); uint32 words (packed bits, bit masks) as the int32 the kernels take."""
    x = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x))
    return x.view(torch.int32) if x.dtype == torch.uint32 else x


def _flat(x):
    return x.reshape(-1) if isinstance(x, torch.Tensor) else np.asarray(x).reshape(-1)


STAGE_LIMIT_IN_FLIGHT = 4   # hz_search_io.stage_limit used when several searches share the GPU (profiles/r02_sm_target.md)


def gemm_sm_target_for(num_roots, in_flight, device):
    """SMs each search's library GEMMs should be sized for when `in_flight` independent searches of `num_roots` trees
    share a GPU.  cuBLASLt sizes a GEMM to fill the whole device, so the GEMMs of different streams queue behind one
    another; with small root batches it pays to size each for a share of the SMs so that they run side by side.
    Measured on B200 (profiles/r02_sm_target.md): 3n/64 SMs up to 56 (24 at 512 trees, 48 at 1024, 56 at 1536-2048);
    from ~3000 trees on the whole-device kernels are the best choice (returns 0)."""
    if in_flight <= 1 or num_roots >= 3072:
        return 0
    sms = torch.cuda.get_device_properties(device).multi_processor_count
    return int(max(16, min(3 * num_roots // 64, 56 * sms // 148)))


ROWS_MIN_BLOCKS_SMALL = 48   # row blocks in flight from which Hanabi-Small gains from the row executor (B200, measured)


def network_executor_for(model, num_roots, in_flight):
    """The network executor executor="auto" picks for `in_flight` independent searches (SearchPipeline slots,
    SelfPlayPool engines) of `num_roots` trees each.  One search at a time: the library chain, whose latency is lower.
    Searches in flight: the row-block resident executor, which holds num_roots / 128 SMs per search instead of the whole
    device.  For the Hanabi-Small network its longer chain (37 us against 15-24 us) only pays once the searches in
    flight keep at least ROWS_MIN_BLOCKS_SMALL 128-row blocks going: measured on B200 (profiles/r03_rowchain_small.md),
    512 trees x 8 and 1024 x 4 in flight (32 blocks) run 11-21 % faster on the library chain, 768 x 8 and 512 x 12
    (48 blocks) 4-13 % slower.  Plans the row executor does not cover (fp32) run the library chain whatever this says."""
    if in_flight <= 1:
        return "library"
    if not getattr(model, "full", True) and in_flight * -(-int(num_roots) // 128) < ROWS_MIN_BLOCKS_SMALL:
        return "library"
    return "rows"


class WaveSchedule:
    """Ticket bookkeeping of SearchPipeline(wave=G): the slot and position each submit takes, and when the wave that
    is still taking tickets ("open") must launch.  Slots are used round robin; ticket id = slot * G + position."""

    def __init__(self, wave, depth):
        self.wave, self.depth = int(wave), int(depth)
        self.open = None      # dict(slot, noisy, fraction, count) of the open wave
        self._next = 0

    def closes(self, noisy, fraction):
        """True when a ticket of this kind cannot join the open wave: one wave is one Roots.prepare call, so the
        noise-ness and (with noise) the exploration fraction must match."""
        return self.open is not None and (self.open["noisy"], self.open["fraction"]) != (noisy, fraction)

    def take(self, noisy, fraction):
        """(slot, position) of the next ticket; opens a wave on the next slot when none is open (position 0)."""
        if self.open is None:
            self.open = dict(slot=self._next, noisy=noisy, fraction=fraction, count=0)
            self._next = (self._next + 1) % self.depth
        p = self.open["count"]
        self.open["count"] += 1
        return self.open["slot"], p

    def full(self):
        return self.open is not None and self.open["count"] == self.wave

    def close(self):
        """The open wave (to launch now); none is open afterwards."""
        w, self.open = self.open, None
        return w

    def slot_of(self, ticket):
        return ticket // self.wave

    def is_open(self, slot):
        return self.open is not None and self.open["slot"] == slot


class SearchPipeline:
    """Searches kept in flight: `depth` slots, each with its own tree batch (and therefore its own captured search
    graph, network buffers and staging buffers) and its own compute stream.  Inputs are copied in on a copy stream and
    root statistics copied out on another, so for host-fed searches the copies of search i+1 / i-1 overlap search i —
    and, because a search is a dependent chain of short launches that leaves the GPU idle at every kernel boundary, the
    searches of different slots overlap each other: independent root batches (the reference's actors, each with its
    own p_mcts_num roots, core/selfplay_worker.py:93,102) fill one another's bubbles.

        pipe = SearchPipeline(MCTS(cfg), model, num_roots, num_actions)
        t = pipe.submit(fraction, noises, rewards, logits, legal, hidden_roots, out_visits, out_values)   # returns at once
        ...
        pipe.wait(t)          # out_visits / out_values now hold the result of that search

    Inputs are what Roots.prepare + MCTS.run_multi take (core/selfplay_worker.py:276-283): pinned host tensors
    (pageable memory works but serialises the copies) or device tensors; outputs likewise.  Device tensors that already
    have the staging buffers' type (float32 / int32 legal mask, contiguous, on this device) are read in place — keep
    them unchanged until wait(ticket).  `noises=None` selects prepare_no_noise.  `gather` (dist.AsyncStatsGather with
    depth >= this depth) additionally all-gathers every search's statistics over the ranks, off the compute streams;
    `gathered(t)` returns them.  Weights must not change while searches are in flight: call drain() before updating
    the module.

    With depth > 1 the network runs on the row-block resident executor (`executor`, hz_rowchain: one launch per
    simulation on n/128 SMs; profiles/r02_rowchain.md, r03_rowchain_small.md) where the plan supports it and, for
    Hanabi-Small, where enough row blocks are in flight for it to pay (network_executor_for).  For the library chain two settings
    make the slots share the GPU instead of queueing (profiles/r02_sm_target.md): `gemm_sm_target`
    (default gemm_sm_target_for(num_roots, depth)) sizes each search's library GEMMs for a share of the SMs, and
    `stage_limit` (default 4) keeps the tree step's shared-memory footprint small enough to sit next to a GEMM CTA.
    Results per search are those of MCTS.run_multi with the same two settings (the SM target changes the rounding of
    the network outputs in the last bits, the staging limit changes nothing).

    Waves (`wave` = G > 1): a slot holds G tickets of `num_roots` trees each and searches them together as ONE batch of
    G * num_roots trees — one input pack (hz_wave_pack), one graph launch, one statistics kernel, one output scatter
    (hz_wave_unpack) and, with `gather`, one all-gather per wave instead of one of each per ticket.  Trees never
    interact, so each ticket gets exactly its own rows back: on the row-block executor they equal, bit for bit, a
    stand-alone Roots(num_roots) + run_multi of that ticket alone; on the library chain, where cuBLASLt may pick other
    kernels for G * num_roots rows, they equal one run_multi over the concatenated batch.  submit() returns the ticket
    id slot * G + position (the slot index for G = 1).  A wave launches when its G-th ticket arrives, on flush(), or
    when wait / stats / gathered names one of its tickets; a submit whose exploration fraction or noise-ness (noises vs
    None) differs from the open wave's launches the open wave first.  A partial wave runs the full-size search with
    padding roots (no legal action) in its unused positions.  Inputs that are already float32 / int32 legal mask / the
    hidden-state pool's dtype, contiguous and on this device or in page-locked host memory are read by the pack kernel
    in place (keep them unchanged until wait(ticket)); outputs of that kind are written in place.  Anything else is
    converted by torch on the caller's stream first, or copied out after the scatter: the slow path.  The executor and
    SM-target rules see the wave's G * num_roots trees.  Waves of 4096 trees need only 7-8 slots in flight, so unlike
    depth-20 pipelines of small searches they need no CUDA_DEVICE_MAX_CONNECTIONS above its default of 8.

    Observation tickets (`stack` = frames per root, `mdp` = "global" or "local"): submit_observations() hands in
    stacked observations instead of the representation network's outputs, and the slot runs the root inference itself
    (InitialPlan, one pack launch hz_obs_pack in place of hz_wave_pack).  A wave holds one kind of ticket.  Observation
    tickets may hand in frame windows of consecutive positions (`positions`) and ask for policy targets (`out_policy`):
    the reanalyze pipeline (reanalyze.ReanalyzePipeline).  A third kind, episode tickets, reads those windows from an
    EpisodeStore in device memory (hz_obs_pack_episodes; ReanalyzePipeline.submit_episodes).

    Waves fill only when a caller submits tickets ahead of its waits: a wait / stats / gathered on a ticket of the open
    wave launches it with the tickets it holds so far, so submit-then-wait per ticket runs waves of one ticket.  Ticket
    ids are reused round robin: consume a ticket before `depth` more waves open (wait with a lag below depth * G
    tickets), or the id names the slot's newer wave: wait() then launches that wave early, and stats() / gathered()
    return the newer wave's rows (as for G = 1, a slot's statistics are valid until it is submitted again).  The
    pipeline is not thread-safe: callers on several threads need one lock around every call (submit, wait, stats,
    gathered, flush, drain)."""

    def __init__(self, mcts, model, num_roots, num_actions, depth=8, device=None, gather=None, gemm_sm_target=None,
                 stage_limit=None, executor="auto", wave=1, stack=None, mdp="global"):
        self.mcts, self.model = mcts, model
        self.depth = int(depth)
        self.wave = int(wave)
        if not 1 <= self.wave <= 64:
            raise ValueError("wave must be 1..64 tickets")
        rows = self.wave * int(num_roots)   # trees per slot
        # "rows": the network as one row-block resident launch per simulation (BoundChain.set_executor) — a quarter of
        # the SMs per search at 4096 trees, which is what searches in flight want; "library": seven (Hanabi-Full) or
        # five (Hanabi-Small) cuBLASLt launches, the lower latency for a search that runs alone.  "auto": see
        # network_executor_for (plans the row executor does not cover fall back to the library chain inside MCTS).
        self.executor = network_executor_for(model, rows, self.depth) if executor == "auto" else executor
        self.n, self.a, self.depth = int(num_roots), int(num_actions), int(depth)
        device = next(model.parameters()).device if device is None else device
        # always indexed ("cuda" -> "cuda:<current>"): tensors report indexed devices, and inputs / outputs are matched
        # against this one to be read or written in place
        self.device = torch.device("cuda", cytree._device_index(device))
        dev, sims = self.device, int(mcts.config.num_simulations)
        if gemm_sm_target is None:
            gemm_sm_target = gemm_sm_target_for(rows, self.depth, dev)
        self.gemm_sm_target = int(gemm_sm_target)
        # searches in flight: a small staging region lets the tree step share SMs with the other slots' GEMM CTAs
        self.stage_limit = (STAGE_LIMIT_IN_FLIGHT if self.depth > 1 else 0) if stage_limit is None else int(stage_limit)
        mcts.max_cached_workspaces = max(mcts.max_cached_workspaces, self.depth + 4)   # one workspace (graph) per slot
        if gather is not None and gather.depth < self.depth:
            raise ValueError("gather.depth must be at least the pipeline depth")
        if gather is not None and gather.n != rows:
            raise ValueError("gather.n must be wave * num_roots (the trees of one slot)")
        self.gather = gather
        self.copy_in, self.copy_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        self.slots = []
        for _ in range(self.depth):
            self.slots.append(dict(
                roots=cytree.Roots(rows, self.a, sims, device=dev), stream=torch.cuda.Stream(dev),
                noise=torch.empty(rows, self.a, device=dev), reward=torch.empty(rows, device=dev),
                logits=torch.empty(rows, self.a, device=dev), legal=torch.empty(rows, self.a, dtype=torch.int32, device=dev),
                hidden=None, stats=None, visits=None, values=None, ticket=None,
                ev_in=torch.cuda.Event(), ev_done=torch.cuda.Event(), ev_out=torch.cuda.Event(), busy=False))
        for s in self.slots:
            # one int32 buffer [n * A visit counts | n value bit patterns]: the statistics kernel writes both parts in
            # place and the all-gather ships the buffer as it is (no packing kernels)
            s["stats"] = torch.empty(rows * (self.a + 1), dtype=torch.int32, device=dev)
            s["visits"] = s["stats"][:rows * self.a].view(rows, self.a)
            s["values"] = s["stats"][rows * self.a:].view(torch.float32)
            if self.wave > 1 or stack is not None:
                # the open wave: its tickets' table entries, the inputs they point at, slow-path outputs, and one
                # caller-stream event per ticket that the slot's stream waits for at launch
                s.update(table=[], keep=[], post=[], ev_tickets=[torch.cuda.Event() for _ in range(self.wave)],
                         kind="hidden", obs_table=[], positions=1, policy_table=[], policy=None, stores=[])
        self._next = 0
        self._waves = WaveSchedule(self.wave, self.depth)
        self._hidden_shape = None    # wave > 1: (feature, pool dtype) of the root hidden states
        self.stack, self._iplan = None if stack is None else int(stack), None
        if self.stack is not None:
            # observation tickets: the frame layout of the network's input, and per slot the root inference's own
            # buffers and cuBLASLt plan (InitialPlan.bound with the slot's tree batch as owner), sized for the wave
            from .hanabi_env import frame_layout
            self.frame_dim, self.frame_words, bit_offset = frame_layout(
                "Hanabi-Full" if getattr(model, "full", True) else "Hanabi-Small", mdp, dev)
            amp = getattr(mcts.config, "amp_type", "none") == "torch_amp"
            self._iplan = model.initial_plan(torch.float16 if amp else torch.float32, self.frame_dim, self.stack)
            self._layout = _lib.ObsLayout(self.stack, self.frame_dim, self._iplan.frame_stride,
                                          self._iplan.dtype.itemsize, self.frame_words, bit_offset)
            self._zero_reward = torch.zeros(rows, device=dev)   # the root reward of initial_inference is 0
            for s in self.slots:
                s["ibound"] = self._iplan.bound(rows, owner=s["roots"])
                if self.gemm_sm_target:
                    check(self._iplan.lib.hz_gemm_plan_set_sm_target(s["ibound"].handle, self.gemm_sm_target))
        self.host_seconds, self.submitted = 0.0, 0

    def submit(self, fraction, noises, rewards, logits, legal, hidden_roots, out_visits=None, out_values=None):
        if self.wave > 1:
            return self._submit_to_wave(fraction, noises, rewards, logits, legal, hidden_roots, out_visits, out_values)
        i = self._next
        self._next = (i + 1) % self.depth
        s = self.slots[i]
        if s["busy"]:
            s["ev_out"].synchronize()          # the slot's previous search has been read out
        s["busy"] = True
        t_host = time.perf_counter()
        hidden_roots = torch.as_tensor(hidden_roots)
        if s["hidden"] is None or s["hidden"].shape != hidden_roots.shape or s["hidden"].dtype != hidden_roots.dtype:
            s["hidden"] = torch.empty(hidden_roots.shape, dtype=hidden_roots.dtype, device=self.device)
        caller = torch.cuda.current_stream(self.device)
        compute = s["stream"]
        if self.gather is not None and s["ticket"] is not None and self.gather.stream is not None:
            # the slot's statistics buffer is the send buffer of its previous all-gather: the new search may only
            # overwrite it once that collective is done
            compute.wait_event(self.gather.slots[s["ticket"]]["done"])
        inputs = dict(noise=noises, reward=rewards, logits=logits, legal=legal, hidden=hidden_roots)
        if all(v is None or self._usable_in_place(v, s[k]) for k, v in inputs.items()):
            # device-resident inputs of the staging buffers' own type: read in place, no copies (the caller keeps them
            # unchanged until wait(ticket)); the slot's stream only has to follow whatever produced them
            compute.wait_stream(caller)
            src = inputs
        else:
            self.copy_in.wait_stream(caller)
            with torch.cuda.stream(self.copy_in):
                # the slot's staging buffers were last read by its previous search, which ev_out (waited above) follows
                if noises is not None:
                    s["noise"].copy_(torch.as_tensor(noises), non_blocking=True)
                s["reward"].copy_(torch.as_tensor(rewards), non_blocking=True)
                s["logits"].copy_(torch.as_tensor(logits), non_blocking=True)
                s["legal"].copy_(torch.as_tensor(legal), non_blocking=True)
                s["hidden"].copy_(hidden_roots, non_blocking=True)
                s["ev_in"].record(self.copy_in)
            compute.wait_event(s["ev_in"])
            src = s
        with torch.cuda.stream(compute):
            if noises is not None:
                s["roots"].prepare(fraction, src["noise"], src["reward"], src["logits"], src["legal"])
            else:
                s["roots"].prepare_no_noise(src["reward"], src["logits"], src["legal"])
            self.mcts.run_multi(s["roots"], self.model, src["hidden"], gemm_sm_target=self.gemm_sm_target,
                                stage_limit=self.stage_limit, executor=self.executor)
            check(s["roots"]._lib.hz_trees_root_stats(s["roots"].handle, compute.cuda_stream, ptr(s["visits"]),
                                                      ptr(s["values"])))
            s["ev_done"].record(compute)
            if self.gather is not None:
                s["ticket"] = self.gather.submit_flat(s["stats"])
        self.copy_out.wait_event(s["ev_done"])
        with torch.cuda.stream(self.copy_out):
            if out_visits is not None:
                out_visits.copy_(s["visits"], non_blocking=True)
            if out_values is not None:
                out_values.copy_(s["values"], non_blocking=True)
            s["ev_out"].record(self.copy_out)
        self.host_seconds += time.perf_counter() - t_host   # host time spent enqueueing (not waiting for the GPU)
        self.submitted += 1
        return i

    def _usable_in_place(self, x, like):
        return (isinstance(x, torch.Tensor) and x.device == like.device and x.dtype == like.dtype and x.shape == like.shape
                and x.is_contiguous())

    def _submit_to_wave(self, fraction, noises, rewards, logits, legal, hidden_roots, out_visits, out_values):
        t_host = time.perf_counter()
        noisy = noises is not None
        fraction = float(fraction) if noisy else 0.0
        if self._waves.closes(noisy, fraction) or self._open_kind() not in (None, "hidden"):
            self._launch_wave()
        hidden_roots = torch.as_tensor(hidden_roots)
        if self._hidden_shape is None:
            feature = int(hidden_roots.shape[-1])
            hidden_shape = (feature, self.mcts.pool_dtype(self.model, feature, self.device))
        else:
            hidden_shape = self._hidden_shape
        feature, hdtype = hidden_shape
        # every input converted and every output checked BEFORE the ticket takes a position: a bad argument raises here
        # and leaves the open wave as it was
        n, a, held = self.n, self.a, []
        rec = _lib.WaveTicket()
        rec.noise = self._wave_input(noises, torch.float32, (n, a), held)
        rec.reward = self._wave_input(rewards, torch.float32, (n,), held)
        rec.logits = self._wave_input(logits, torch.float32, (n, a), held)
        rec.legal = self._wave_input(legal, torch.int32, (n, a), held)
        rec.hidden = self._wave_input(hidden_roots, hdtype, (n, feature), held)
        in_place = [self._wave_output(x, dtype, shape) for x, dtype, shape in
                    ((out_visits, torch.int32, (n, a)), (out_values, torch.float32, (n,)))]
        self._hidden_shape = hidden_shape
        return self._join("hidden", noisy, fraction, rec, None, held, in_place, out_visits, out_values, t_host)

    def _open_kind(self):
        """Kind of ticket ("hidden", "obs" or "episodes") the open wave holds, None when no wave is open."""
        return None if self._waves.open is None else self.slots[self._waves.open["slot"]]["kind"]

    def _open_reads(self, store):
        """True when the open wave holds a ticket that reads `store` (an EpisodeStore)."""
        return self._open_kind() == "episodes" and any(
            st is store for st, _, _ in self.slots[self._waves.open["slot"]]["stores"])

    def _join(self, kind, noisy, fraction, rec, obs_rec, held, in_place, out_visits, out_values, t_host, positions=1,
              policy=None, store=None):
        """The ticket takes the next position of the open wave (opening one if needed), launching it when full.
        policy: (policy_mask address, out_policy) of an observation ticket that asked for policy targets.
        store: (EpisodeStore, lowest id read, the store's newest add event or None) of an episode ticket."""
        n = self.n
        if self.wave == 1:
            self._waves._next = self._next      # submit() and observation tickets share the round robin over slots
        i, p = self._waves.take(noisy, fraction)
        if self.wave == 1:
            self._next = self._waves._next
        s = self.slots[i]
        if p == 0:
            if s["busy"]:
                t_wait = time.perf_counter()
                s["ev_out"].synchronize()   # the slot's previous wave has been read out
                t_host += time.perf_counter() - t_wait   # waiting for the GPU is not host time
            s["busy"] = True
            s["table"], s["keep"], s["post"], s["obs_table"], s["kind"] = [], [], [], [], kind
            s["positions"], s["policy_table"], s["stores"] = positions, [], []
        if store is not None:
            s["stores"].append(store)
        s["keep"] += held                   # alive until the slot is reused
        rows = slice(p * n, (p + 1) * n)
        for out, ok, buf in zip((out_visits, out_values), in_place, (s["visits"], s["values"])):
            if out is not None and not ok:
                s["post"].append((out, buf[rows]))
        if obs_rec is not None:
            prec = None
            if policy is not None:
                mask, out_policy = policy
                if self._writable_policy(out_policy):
                    prec = _lib.PolicyTicket(mask=mask, out=ptr(out_policy))
                else:      # slow path: the slot's own rows, copied out after the policy launch
                    prec = _lib.PolicyTicket(mask=mask, out=ptr(self._policy_rows(s)[rows]))
                    s["post"].append((out_policy, s["policy"][rows]))
            s["policy_table"].append(prec)
        rec.out_visits = ptr(out_visits) if in_place[0] else None
        rec.out_values = ptr(out_values) if in_place[1] else None
        s["table"].append(rec)
        if obs_rec is not None:
            s["obs_table"].append(obs_rec)
        s["ev_tickets"][p].record(torch.cuda.current_stream(self.device))   # after whatever produced the inputs
        if self._waves.full():
            self._launch_wave()
        self.host_seconds += time.perf_counter() - t_host
        self.submitted += 1
        return i * self.wave + p    # ticket id

    def submit_observations(self, fraction, noises, obs, legal, out_visits=None, out_values=None, positions=1,
                            policy_mask=None, out_policy=None):
        """A search that starts from stacked observations (core/selfplay_worker.py:258-283: stack_obs ->
        initial_inference -> prepare -> run_multi) instead of the representation network's outputs; needs a pipeline
        built with `stack` (frames per root) and `mdp` ("global" or "local" observations).  The root inference runs in
        the slot (InitialPlan of the model, fp16 for amp_type "torch_amp"), the root reward is 0, and the results are
        those of submit() with the hidden states, logits and legal mask that inference gives.  Returns a ticket id as
        submit() does; a ticket of the other kind (submit) launches the open wave first, as a change of noise-ness does.

        obs: the frames of every root, oldest first, as float32 or uint8 0/1 values [n, stack, D] (or [n, stack * D]),
        or as packed bits: int32 [n, stack, W] (or [n, stack * W]), each frame the W-word string that step_bits /
        EnvPipeline(fmt="bits") hand out, of which the pack kernel takes the global observation or its local suffix
        (hanabi_env.frame_layout).  legal: int32 or float32 [n, A], or one int32 bit mask word per root ([n]; e.g.
        `meta[:, 0]` of EnvPipeline's meta rows).  noises: float32 [n, A] or None (prepare_no_noise).  Rows may have any
        stride.  Inputs already in one of these forms on this device or in page-locked host memory are read by the
        pack kernel in place: keep them unchanged until wait(ticket).  Anything else is converted by torch on the
        caller's stream first.  Outputs as for submit().  Weights: drain() before updating the module.

        Frame windows (`positions` = P > 1, the reanalyze batch, whose consecutive positions share frames): obs holds
        n / P windows of S + P - 1 frames, [n / P, S + P - 1, D] (or [n / P, (S + P - 1) * D]; bits likewise with W),
        and root i * P + p takes frames p .. p + S - 1 of window i; legal moves and noises stay per root.  The pack
        kernel expands the windows on the device (hz_obs_pack_windows), so the caller hands in one window per sample
        instead of P stacks (it still reads a frame once for every stack that holds it).  A wave holds tickets of one
        P: a different P launches the open wave first.
        Policy targets (`out_policy`, float64 of n * A elements): the visit counts turned into hz_visit_policy's
        correctly rounded quotients, all-zero rows where `policy_mask` (uint8 [n], None keeps every row) is 0, by one
        launch per wave after the statistics scatter (hz_wave_policy).  out_policy is written in place when it is
        contiguous on this device or in page-locked host memory, else copied after the wave; the mask is read in place
        under the same rule, else converted."""
        if self._iplan is None:
            raise RuntimeError("submit_observations needs a pipeline built with stack= (the frame layout)")
        t_host = time.perf_counter()
        noisy = noises is not None
        fraction = float(fraction) if noisy else 0.0
        n, a, held = self.n, self.a, []
        positions = int(positions)
        if positions < 1 or n % positions:
            raise ValueError(f"positions = {positions} must be >= 1 and divide the {n} roots of a ticket")
        # every input and output checked, then converted, BEFORE the ticket takes a position
        obs, ofmt, odtype, oshape, odense = self._obs_form(obs, positions)
        legal, lfmt, ldtype, lshape, ldense = self._legal_form(legal)
        if noises is not None and _as_tensor(noises).numel() != n * a:
            raise ValueError(f"noises must hold [{n}, {a}] values, got {tuple(_as_tensor(noises).shape)}")
        in_place = [self._wave_output(x, dtype, shape) for x, dtype, shape in
                    ((out_visits, torch.int32, (n, a)), (out_values, torch.float32, (n,)))]
        if out_policy is None and policy_mask is not None:
            raise ValueError("policy_mask without out_policy")
        if out_policy is not None:
            self._wave_output(out_policy, torch.float64, (n, a))       # raises unless it can take n * A values
            if out_policy.dtype != torch.float64:
                raise ValueError(f"out_policy must be float64, got {out_policy.dtype}")
            if policy_mask is not None:
                policy_mask = _as_tensor(policy_mask)
                if policy_mask.numel() != n:
                    raise ValueError(f"policy_mask must hold {n} values, got {tuple(policy_mask.shape)}")
                policy_mask = policy_mask.reshape(n)
        orec = _lib.ObsTicket()
        orec.obs, orec.ld_obs = self._source(obs, odtype, oshape, odense, held)
        orec.legal, orec.ld_legal = self._source(legal, ldtype, lshape, ldense, held)
        orec.noise = self._wave_input(noises, torch.float32, (n, a), held)
        orec.obs_format, orec.legal_format = ofmt, lfmt
        policy = None if out_policy is None else (self._wave_input(policy_mask, torch.uint8, (n,), held), out_policy)
        if (self._waves.closes(noisy, fraction) or self._open_kind() not in (None, "obs")
                or (self._open_kind() == "obs" and self.slots[self._waves.open["slot"]]["positions"] != positions)):
            self._launch_wave()
        return self._join("obs", noisy, fraction, _lib.WaveTicket(), orec, held, in_place, out_visits, out_values,
                          t_host, positions, policy)

    def _submit_episodes(self, fraction, noises, store, samples, low_id, out_policy):
        """An observation ticket of frame windows read from an EpisodeStore (reanalyze.ReanalyzePipeline
        .submit_episodes): `samples` is hz_obs_pack_episodes' int32 [n / P, 4] on this device (P = positions), low_id
        the lowest episode id it names, noises float32 [n, A] on this device (masked by the legal rows in the pack) or
        None, out_policy float64 of n * A elements (its targets; rows past an episode's end zero).  The checks against
        the store are the caller's; the pack waits for the store's adds made so far, and the store is told about the
        pack (reader event) and about this pipeline (an evicting add launches the open wave first).  A wave holds
        tickets of one kind and one P."""
        if self._iplan is None:
            raise RuntimeError("episode tickets need a pipeline built with stack= (the frame layout)")
        t_host = time.perf_counter()
        noisy = noises is not None
        fraction = float(fraction) if noisy else 0.0
        n, a, held = self.n, self.a, [samples]
        positions = n // samples.shape[0]
        self._wave_output(out_policy, torch.float64, (n, a))       # raises unless it can take n * A values
        if out_policy.dtype != torch.float64:
            raise ValueError(f"out_policy must be float64, got {out_policy.dtype}")
        mask = torch.empty(n, dtype=torch.uint8, device=self.device)   # written by the pack, read by hz_wave_policy
        held.append(mask)
        rec = _lib.EpisodeTicket(frames=ptr(store.frames), ld_frames=store.frames.stride(0), legal=ptr(store.legal),
                                 samples=ptr(samples), noise=self._wave_input(noises, torch.float32, (n, a), held),
                                 mask=ptr(mask))
        if (self._waves.closes(noisy, fraction) or self._open_kind() not in (None, "episodes")
                or (self._open_kind() == "episodes" and self.slots[self._waves.open["slot"]]["positions"] != positions)):
            self._launch_wave()
        store._watch(self)
        return self._join("episodes", noisy, fraction, _lib.WaveTicket(), rec, held, [False, False], None, None, t_host,
                          positions, (ptr(mask), out_policy), store=(store, int(low_id), store._last_add))

    def _writable_policy(self, x):
        """True when hz_wave_policy can write `out_policy` itself (contiguous float64 here or in page-locked memory)."""
        return x.dtype == torch.float64 and x.is_contiguous() and (
            x.device == self.device or (x.device.type == "cpu" and x.is_pinned()))

    def _policy_rows(self, s):
        """The slot's float64 [wave * n, A] policy buffer: slow-path outputs and the rows of tickets without targets."""
        if s["policy"] is None:
            s["policy"] = torch.empty(self.wave * self.n, self.a, dtype=torch.float64, device=self.device)
        return s["policy"]

    def _obs_form(self, x, positions=1):
        """(tensor, HZ_OBS_* format, dtype the kernel reads, shape, frames dense in the row) of a ticket's frames:
        n / positions rows of stack + positions - 1 frames."""
        n, S = self.n // positions, self.stack + positions - 1
        x = _as_tensor(x)
        if x.dtype == torch.int32:
            fmt, width, dtype = _lib.HZ_OBS_BITS, self.frame_words, torch.int32
        elif x.dtype == torch.uint8:
            fmt, width, dtype = _lib.HZ_OBS_U8, self.frame_dim, torch.uint8
        else:
            fmt, width, dtype = _lib.HZ_OBS_F32, self.frame_dim, torch.float32
        if tuple(x.shape) not in ((n, S, width), (n, S * width)):
            raise ValueError(f"obs must be [{n}, {S}, {width}] or [{n}, {S * width}] ({x.dtype}), got {tuple(x.shape)}")
        return x, fmt, dtype, (n, S * width), x.stride(-1) == 1 and (x.dim() == 2 or x.stride(1) == width)

    def _legal_form(self, x):
        """(tensor, HZ_LEGAL_* format, dtype the kernel reads, shape, row dense) of a ticket's legal moves."""
        n, a = self.n, self.a
        x = _as_tensor(x)
        if x.dim() == 1:
            if x.shape[0] != n or x.dtype != torch.int32:
                raise ValueError(f"a legal bit mask must be int32 [{n}], got {x.dtype} {tuple(x.shape)}")
            return x, _lib.HZ_LEGAL_MASK, torch.int32, (n,), True      # one word per root at any row stride
        if tuple(x.shape) != (n, a):
            raise ValueError(f"legal must be [{n}, {a}] or an int32 bit mask [{n}], got {tuple(x.shape)}")
        if x.dtype == torch.float32:
            return x, _lib.HZ_LEGAL_F32, torch.float32, (n, a), x.stride(-1) == 1
        return x, _lib.HZ_LEGAL_I32, torch.int32, (n, a), x.stride(-1) == 1

    def _source(self, x, dtype, shape, dense, held):
        """(address, row stride in elements) the pack kernel reads `x` at: in place when it has the kernel's type and
        layout on this device or in page-locked host memory, else converted by torch on the caller's stream."""
        if not (x.dtype == dtype and dense and (x.device == self.device or (x.device.type == "cpu" and x.is_pinned()))):
            x = cytree.as_device(x, dtype, self.device, shape)      # slow path
        held.append(x)
        return x.data_ptr(), x.stride(0)

    def _readable_in_place(self, x, dtype, shape):
        return (isinstance(x, torch.Tensor) and x.dtype == dtype and tuple(x.shape) == shape and x.is_contiguous()
                and (x.device == self.device or (x.device.type == "cpu" and x.is_pinned())))

    def _wave_input(self, x, dtype, shape, held):
        """Address the pack kernel reads a ticket input from (None -> NULL); the tensor read is appended to `held`."""
        if x is None:
            return None
        if not self._readable_in_place(x, dtype, shape):
            x = cytree.as_device(x, dtype, self.device, shape)     # slow path: torch converts on the caller's stream
        held.append(x)
        return x.data_ptr()

    def _wave_output(self, x, dtype, shape):
        """True when the scatter kernel can write a ticket output in place; False for the slow path (a torch copy after
        the scatter).  An output that cannot take the ticket's rows raises."""
        if x is None:
            return False
        if not isinstance(x, torch.Tensor) or x.numel() != int(np.prod(shape)):
            raise ValueError(f"outputs must be tensors of {int(np.prod(shape))} elements {shape}")
        return self._readable_in_place(x, dtype, shape)

    def _launch_wave(self):
        """Search the open wave: pack -> prepare -> run_multi -> root statistics -> (all-gather) -> scatter, all on
        the slot's stream after the events its tickets recorded on their callers' streams."""
        w = self._waves.close()
        s = self.slots[w["slot"]]
        roots, compute, count = s["roots"], s["stream"], len(s["table"])
        lib, dev = roots._lib, roots.device_index
        for ev in s["ev_tickets"][:count]:
            compute.wait_event(ev)
        for _, _, ev in s["stores"]:
            if ev is not None:
                compute.wait_event(ev)       # the episode store's adds made before the ticket was submitted
        if self.gather is not None and s["ticket"] is not None and self.gather.stream is not None:
            compute.wait_event(self.gather.slots[s["ticket"]]["done"])   # the stats buffer was its send buffer
        table = (_lib.WaveTicket * count)(*s["table"])
        st = compute.cuda_stream
        with torch.cuda.stream(compute):
            if s["kind"] != "hidden":
                b = s["ibound"]
                noise = ptr(s["noise"]) if w["noisy"] else None
                otab = ((_lib.ObsTicket if s["kind"] == "obs" else _lib.EpisodeTicket) * count)(*s["obs_table"])
                if s["kind"] == "episodes":
                    check(lib.hz_obs_pack_episodes(st, dev, otab, count, self.wave, self.n, self.a,
                                                   _lib.C.byref(self._layout), s["positions"], ptr(b.x),
                                                   ptr(s["legal"]), noise))
                    read = torch.cuda.Event()
                    read.record(compute)         # an add that evicts what this pack read waits for it
                    for store, low, _ in s["stores"]:
                        store._read(read, low)
                elif s["positions"] > 1:
                    check(lib.hz_obs_pack_windows(st, dev, otab, count, self.wave, self.n, self.a,
                                                  _lib.C.byref(self._layout), s["positions"], ptr(b.x), ptr(s["legal"]),
                                                  noise))
                else:
                    check(lib.hz_obs_pack(st, dev, otab, count, self.wave, self.n, self.a, _lib.C.byref(self._layout),
                                          ptr(b.x), ptr(s["legal"]), noise))
                recurrent = self.mcts._plan(self.model)
                if self._iplan.refresh() | bool(recurrent is not None and recurrent.refresh()):
                    # the weights were re-folded on this stream; the other slots' streams read them too
                    compute.synchronize()
                hidden, reward = self._iplan.run_bound(b, s["logits"]), self._zero_reward
            else:
                if s["hidden"] is None:
                    feature, hdtype = self._hidden_shape
                    s["hidden"] = torch.empty(self.wave * self.n, feature, dtype=hdtype, device=self.device)
                check(lib.hz_wave_pack(st, dev, table, count, self.wave, self.n, self.a,
                                       s["hidden"].shape[1] * s["hidden"].element_size(),
                                       ptr(s["noise"]) if w["noisy"] else None, ptr(s["reward"]), ptr(s["logits"]),
                                       ptr(s["legal"]), ptr(s["hidden"])))
                hidden, reward = s["hidden"], s["reward"]
            if w["noisy"]:
                roots.prepare(w["fraction"], s["noise"], reward, s["logits"], s["legal"])
            else:
                roots.prepare_no_noise(reward, s["logits"], s["legal"])
            self.mcts.run_multi(roots, self.model, hidden, gemm_sm_target=self.gemm_sm_target,
                                stage_limit=self.stage_limit, executor=self.executor)
            check(lib.hz_trees_root_stats(roots.handle, st, ptr(s["visits"]), ptr(s["values"])))
            s["ev_done"].record(compute)
            if self.gather is not None:
                s["ticket"] = self.gather.submit_flat(s["stats"])
            check(lib.hz_wave_unpack(st, dev, table, count, self.wave, self.n, self.a, ptr(s["stats"])))
            if s["kind"] != "hidden" and any(r is not None for r in s["policy_table"]):
                # tickets without policy targets write theirs into the slot's own rows (the kernel takes no NULL output)
                prows = [r if r is not None else
                         _lib.PolicyTicket(mask=None, out=ptr(self._policy_rows(s)[k * self.n:(k + 1) * self.n]))
                         for k, r in enumerate(s["policy_table"])]
                check(lib.hz_wave_policy(st, dev, (_lib.PolicyTicket * count)(*prows), count, self.wave, self.n,
                                         self.a, ptr(s["stats"])))
            for out, rows in s["post"]:
                out.copy_(rows.reshape(out.shape), non_blocking=True)
            s["ev_out"].record(compute)

    def flush(self):
        """Launch the open wave now, with however many tickets it holds (nothing to do for wave = 1)."""
        if self._waves.open is not None:
            t_host = time.perf_counter()
            self._launch_wave()
            self.host_seconds += time.perf_counter() - t_host

    def _slot_of(self, ticket):
        """Slot of a ticket; launches the ticket's wave if it is still open."""
        slot = self._waves.slot_of(ticket)
        if self._waves.is_open(slot):
            self.flush()
        return slot

    def wait(self, ticket):
        self.slots[self._slot_of(ticket)]["ev_out"].synchronize()

    def stats(self, ticket):
        """Device tensors (visits int32 [n, A], values float32 [n]) of a ticket's search (its rows of the wave's
        buffer); valid until the slot is submitted again.  The current stream waits for the search."""
        s = self.slots[self._slot_of(ticket)]
        torch.cuda.current_stream(self.device).wait_event(s["ev_done"])
        rows = slice(ticket % self.wave * self.n, (ticket % self.wave + 1) * self.n)
        return s["visits"][rows], s["values"][rows]

    def gathered(self, ticket):
        """All ranks' statistics of a ticket's search (needs `gather`), [world * n, A] and [world * n], ranks in order;
        the current stream waits for the collective."""
        visits, values = self.gather.result(self.slots[self._slot_of(ticket)]["ticket"])
        if self.wave == 1:
            return visits, values
        return wave_rows(visits, values, self.gather.world, self.wave, ticket % self.wave)

    def drain(self):
        self.flush()
        for s in self.slots:
            if s["busy"]:
                s["ev_out"].synchronize()
                s["stream"].synchronize()
                s["busy"] = False
        if self.gather is not None and self.gather.stream is not None:
            self.gather.stream.synchronize()
