"""Reanalyze caller of the search — SURVEY.md §8f row N4.

`reanalyze_policies` is the MCTS part of BatchWorker._prepare_policy_re
(/root/reference/core/reanalyze_worker.py:308-371): the learner's target generation re-searches
`batch * (num_unroll_steps + 1)` stored positions with the current target model and turns the root visit
counts into policy targets, all-zero for positions past the end of their trajectory.  Same engine as
self-play (roots with all-zero legal masks included), nothing leaves the device until the targets do.

`ReanalyzePipeline` is its asynchronous form over a SearchPipeline: the caller hands in one window of stored frames
per sampled trajectory (the learner's K + 1 consecutive positions share all but K of their frames), the windows are
expanded into stacks on the device, searches stay in flight, and the policy targets are written by one launch per wave.
With an EpisodeStore (trajectory.py) on the same GPU, `submit_episodes` names each sample as (episode id, start) and the
pack reads the windows from the store's arenas: the frames never cross the host link.
"""
import numpy as np
import torch

from . import _lib, cytree
from ._lib import check, ptr
from .mcts import MCTS, SearchPipeline, _as_tensor
from .selfplay import dirichlet_noise


@torch.no_grad()
def reanalyze_policies(config, model, obs, legal_actions, policy_mask, num_unroll_steps, noises=None, mcts=None,
                       as_tensor=False, noise_seed=0, noise_step=0):
    """obs [B, obs_dim * stack] (float; host or CUDA), legal_actions [B, A] 0/1, policy_mask [B] (0 = position out
    of its trajectory), B = batch * (num_unroll_steps + 1) in trajectory-major order.  `noises` [B, A] replaces
    the Dirichlet draw (the reference multiplies its draw by the legal mask, :343; so is this one); without it the
    draw is selfplay.dirichlet_noise(seed=noise_seed, step=noise_step), reproducible on the host.
    Returns batch_policies_re: float64 [batch, num_unroll_steps + 1, A] (numpy, or a CUDA tensor with as_tensor).
    """
    lib = _lib.load()
    dev = next(model.parameters()).device
    A = int(config.action_space_size) if hasattr(config, "action_space_size") else int(np.shape(legal_actions)[-1])
    obs = cytree.as_device(obs, torch.float32, dev)
    B = obs.shape[0]
    per = int(num_unroll_steps) + 1
    if B % per:
        raise ValueError(f"{B} positions is not a multiple of num_unroll_steps + 1 = {per}")
    legal = cytree.as_device(legal_actions, torch.float32, dev, (B, A))
    mask = cytree.as_device(policy_mask, torch.uint8, dev, (B,))
    model.eval()
    amp = getattr(config, "amp_type", "none") == "torch_amp"
    with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
        _, logits, hidden = model.initial_inference_device(obs)       # :321-336 (value prefix of a root is 0)
    if noises is None:
        noises = dirichlet_noise(B, A, getattr(config, "root_dirichlet_alpha", 0.3), dev, noise_seed, noise_step)
    noises = cytree.as_device(noises, torch.float32, dev, (B, A)) * legal                       # :343
    roots = cytree.Roots(B, A, int(config.num_simulations), device=dev)
    roots.prepare(config.root_exploration_fraction, noises, torch.zeros(B, device=dev), logits.float(), legal.int())
    (mcts or MCTS(config)).run_multi(roots, model, hidden)                                       # :347
    visits = roots.get_distributions_tensor()
    out = torch.empty(B, A, dtype=torch.float64, device=dev)
    check(lib.hz_visit_policy(torch.cuda.current_stream(dev).cuda_stream, ptr(visits), ptr(mask), B, A, ptr(out), None))
    out = out.view(B // per, per, A)
    return out if as_tensor else out.cpu().numpy()


class ReanalyzePipeline:
    """reanalyze_policies with searches in flight: `batch` trajectory windows of `num_unroll_steps` + 1 positions per
    ticket, one SearchPipeline of batch * (num_unroll_steps + 1) roots (`depth` slots, `wave` tickets per search).

        rp = ReanalyzePipeline(config, model, batch, K, stack)
        t = rp.submit(obs_windows, legal_actions, policy_mask, noise_seed=s, noise_step=i)    # returns at once
        ...
        targets = rp.result(t)           # float64 [batch, K + 1, A]

    obs_windows: [batch, K + stack, D] float32 or uint8 0/1 frames, oldest first (a slice of the recorder's flushed
    'o' rows), or packed bit strings int32 [batch, K + stack, W] / [batch, (K + stack) * W]; position p of a sample
    searches frames p .. p + stack - 1.  legal_actions: [batch, K + 1, A] 0/1, or int32 bit-mask words [batch, K + 1].
    policy_mask: [batch, K + 1] (0 = position past the end of its trajectory: an all-zero target row).  Inputs may be
    device or page-locked host tensors, read in place: keep them unchanged until result(ticket).  Frames of masked
    positions past the end of an episode may hold anything; with all-zero legal rows there, the targets do not depend
    on them.  Without `noises` ([batch * (K + 1), A]) the Dirichlet draw is
    dirichlet_noise(batch * (K + 1), A, alpha, seed=noise_seed, step=noise_step) on the caller's stream, the draw
    reanalyze_policies makes; either way it is multiplied by the legal mask, as there.  The exploration fraction is
    config.root_exploration_fraction and the root reward 0.  `out` (float64, batch * (K + 1) * A elements) receives
    the targets; by default a new device tensor.  Results equal a submit_observations of the expanded stacks followed
    by hz_visit_policy; against reanalyze_policies they differ only by the plan's rounding of the root inference.
    Weights: drain() before updating the module.  Not thread-safe, as SearchPipeline."""

    def __init__(self, config, model, batch, num_unroll_steps, stack, mdp="global", depth=8, wave=1, device=None):
        self.config, self.model = config, model
        self.batch, self.per, self.stack = int(batch), int(num_unroll_steps) + 1, int(stack)
        self.a = int(config.action_space_size)
        self.roots = self.batch * self.per
        model.eval()
        self.pipe = SearchPipeline(MCTS(config), model, self.roots, self.a, depth=depth, device=device, wave=wave,
                                   stack=self.stack, mdp=mdp)
        self.device = self.pipe.device
        self._out = {}

    def submit(self, obs_windows, legal_actions, policy_mask, noises=None, noise_seed=0, noise_step=0, out=None):
        B, per, a, dev = self.batch, self.per, self.a, self.device
        legal = _as_tensor(legal_actions)
        if tuple(legal.shape) not in ((B, per, a), (B, per)) or (legal.dim() == 2 and legal.dtype != torch.int32):
            raise ValueError(f"legal_actions must be [{B}, {per}, {a}] or int32 bit masks [{B}, {per}], "
                             f"got {legal.dtype} {tuple(legal.shape)}")
        mask = _as_tensor(policy_mask)
        if tuple(mask.shape) != (B, per):
            raise ValueError(f"policy_mask must be [{B}, {per}], got {tuple(mask.shape)}")
        self.pipe._obs_form(obs_windows, per)          # raises on a wrong window shape before any device work
        if out is None:
            out = torch.empty(B, per, a, dtype=torch.float64, device=dev)
        legal = legal.reshape(self.roots, -1) if legal.dim() == 3 else legal.reshape(self.roots)
        if legal.dim() == 2:
            legal_f = legal.to(device=dev, dtype=torch.float32, non_blocking=True)
        else:       # bit-mask words -> 0/1 rows for the noise mask
            words = legal.to(device=dev, non_blocking=True)
            legal_f = ((words.unsqueeze(1) >> torch.arange(a, device=dev, dtype=torch.int32)) & 1).float()
        if noises is None:
            noises = dirichlet_noise(self.roots, a, getattr(self.config, "root_dirichlet_alpha", 0.3), dev, noise_seed,
                                     noise_step)
        noises = cytree.as_device(noises, torch.float32, dev, (self.roots, a)) * legal_f           # :343
        t = self.pipe.submit_observations(self.config.root_exploration_fraction, noises, obs_windows, legal,
                                          positions=per, policy_mask=mask.reshape(self.roots), out_policy=out)
        self._out[t] = out
        return t

    def submit_episodes(self, store, ids, starts, noises=None, noise_seed=0, noise_step=0, out=None):
        """submit() with the windows read from an EpisodeStore on this device: sample b searches positions
        starts[b] .. starts[b] + K of episode ids[b] (int [batch] each).  Frames are the episode's rows from frame
        starts[b] on, the last frame repeated past its end; positions past the end (start + p >= T) get all-zero legal
        rows and a zero target row.  Only the sample rows (16 bytes a sample) cross from the host.  Targets equal
        submit() of the same windows, legal rows and masks cut from the flushed episodes.  Raises before taking a ticket
        on an evicted or unknown id, a start outside 0..T - 1, or a store whose device, obs_dim, num_actions or stack
        is not the pipeline's.  Noise, `out` and the result as submit()."""
        B, per, a, dev = self.batch, self.per, self.a, self.device
        if (store.device, store.obs_dim, store.num_actions, store.stack) != (dev, self.pipe.frame_dim, a, self.stack):
            raise ValueError(f"store ({store.device}, obs_dim {store.obs_dim}, num_actions {store.num_actions}, stack "
                             f"{store.stack}) does not fit the pipeline ({dev}, obs_dim {self.pipe.frame_dim}, "
                             f"num_actions {a}, stack {self.stack})")
        ids = np.asarray(ids, np.int64).reshape(-1)
        starts = np.asarray(starts, np.int64).reshape(-1)
        if ids.size != B or starts.size != B:
            raise ValueError(f"ids and starts must hold {B} values each, got {ids.size} and {starts.size}")
        samples = store.samples(ids, starts, per)        # raises on evicted ids and bad starts
        if noises is not None and _as_tensor(noises).numel() != self.roots * a:
            raise ValueError(f"noises must hold [{self.roots}, {a}] values, got {tuple(_as_tensor(noises).shape)}")
        if out is None:
            out = torch.empty(B, per, a, dtype=torch.float64, device=dev)
        self.pipe._wave_output(out, torch.float64, (self.roots, a))      # raises before anything is enqueued
        if out.dtype != torch.float64:
            raise ValueError(f"out must be float64, got {out.dtype}")
        if noises is None:
            noises = dirichlet_noise(self.roots, a, getattr(self.config, "root_dirichlet_alpha", 0.3), dev, noise_seed,
                                     noise_step)
        noises = cytree.as_device(noises, torch.float32, dev, (self.roots, a))     # legal-masked in the pack (:343)
        samples = torch.from_numpy(samples).pin_memory().to(dev, non_blocking=True)
        t = self.pipe._submit_episodes(self.config.root_exploration_fraction, noises, store, samples, int(ids.min()), out)
        self._out[t] = out
        return t

    def result(self, ticket):
        """The targets of a ticket, float64 [batch, K + 1, A] (its `out`), once its search is done."""
        self.pipe.wait(ticket)
        return self._out[ticket].view(self.batch, self.per, self.a)

    def drain(self):
        self.pipe.drain()
