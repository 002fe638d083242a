"""Experiment: reanalyze policy targets (SURVEY.md §8f N4) on today's path against ReanalyzePipeline.  Hanabi-Full,
global observation, stack 4, K = num_unroll_steps = 5 (6 positions per sampled window), fp16 (torch_amp), 50
simulations, one GPU, batches of 256 and 682 windows (1536 and 4092 roots per ticket):
  (a) reanalyze_policies, one call at a time, float32 stacks + float legal rows from pinned host memory (returns numpy)
  (b) ReanalyzePipeline, uint8 windows [batch, K + 4, 785] + legal bit-mask words from pinned host memory
  (c) the same pipeline, the windows expanded on the host into uint8 stacks (submit_observations, positions = 1)
  (d) ReanalyzePipeline, packed bit-string windows [batch, (K + 4) * 25]
Pipeline arms write the targets to pinned host memory, as (a) hands them back; waves of about 4096 trees (3 tickets of
1536 roots, 1 of 4092), 8 searches in flight.  Rates count every position (all kept) and 49 simulations per position;
the timed window submits TICKETS tickets and ends with drain() + a synchronise.  Host us per ticket =
SearchPipeline.host_seconds / submitted (for (a) the wall time per call, which includes the wait).  H2D bytes per
position are computed from the shapes each arm hands in.  Then (e): hz_obs_pack_windows alone against hz_obs_pack of
the expanded stacks, CUDA events over many launches.  Writes OUT/r05_reanalyze.jsonl and OUT/r05_reanalyze.md; the card
and its power limit are read in the same run.  Env: OUT (default /tmp/reanalyze), TICKETS (150), CALLS (40), REPS (2)."""
import os
import sys

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes
import json
import statistics
import subprocess
import time
import traceback

import numpy as np
import torch

from hanabizero_b200 import _lib
from hanabizero_b200.hanabi_env import HanabiVecEnv
from hanabizero_b200.mcts import SearchConfig
from hanabizero_b200.model import MuZeroNetFull
from hanabizero_b200.reanalyze import ReanalyzePipeline, reanalyze_policies
from hanabizero_b200.selfplay import dirichlet_noise

OUT = os.environ.get("OUT", "/tmp/reanalyze")
TICKETS = int(os.environ.get("TICKETS", "150"))
CALLS = int(os.environ.get("CALLS", "40"))
REPS = int(os.environ.get("REPS", "2"))
K, STACK, SIMS, A, D, W = 5, 4, 50, 20, 785, 25
PER = K + 1
DEPTH = 8
SHAPES = [(256, 3), (682, 1)]       # (windows per ticket, tickets per wave): waves of 4608 and 4092 trees
INPUTS = 4                          # distinct tickets cycled through
dev = torch.device("cuda")
os.makedirs(OUT, exist_ok=True)
RECS = []


def emit(rec):
    print(json.dumps(rec), flush=True)
    RECS.append(rec)
    with open(os.path.join(OUT, "r05_reanalyze.jsonl"), "a") as f:
        f.write(json.dumps(rec) + "\n")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return dict(device=torch.cuda.get_device_name(0), nvidia_smi=line, torch=torch.__version__)


def config():
    cfg = SearchConfig(num_simulations=SIMS, amp_type="torch_amp")
    cfg.action_space_size = A
    return cfg


def windows(batch, seed):
    """`batch` windows of real Hanabi-Full play (6 random moves, then K + STACK recorded ones): uint8 frames
    [batch, K + STACK, D], packed strings int32 [batch, (K + STACK) * W], legal float [batch, PER, A] of the position
    each stack ends at, all on the host."""
    env = HanabiVecEnv(batch, "Hanabi-Full", np.arange(batch) + seed)
    g, _, legal = env.reset_all()
    gen = torch.Generator(device=dev).manual_seed(seed)
    frames, bits, legals = [], [], []
    for i in range(6 + K + STACK):
        if i >= 6:
            frames.append(g.to(torch.uint8))
            legals.append(legal.clone())
            bits.append(env.step_bits(None)[:, :W].clone())       # the same observation as a packed string
        g, _, legal, _, _, _ = env.step_all(torch.multinomial(legal, 1, generator=gen).view(-1).int(), auto_reset=True)
    env.check()
    u8 = torch.stack(frames, 1).cpu()                                     # [batch, K + STACK, D]
    bits = torch.stack(bits, 1).reshape(batch, -1).cpu()                  # [batch, (K + STACK) * W]
    legal = torch.stack(legals, 1)[:, STACK - 1:].cpu()                   # [batch, PER, A]
    assert torch.equal(torch.from_numpy(np.unpackbits(bits.numpy().view(np.uint8).reshape(batch, K + STACK, 4 * W),
                                                      axis=2, bitorder="little")[:, :, :D]), u8)
    return dict(u8=u8, bits=bits, legal=legal)


def expand(w):
    """[batch, K + STACK, ...] -> [batch * PER, STACK, ...]: position p of a window = its frames p .. p + STACK - 1."""
    return torch.stack([w[:, p:p + STACK] for p in range(PER)], 1).reshape(w.shape[0] * PER, STACK, *w.shape[2:])


def words(legal):
    return ((legal.long() << torch.arange(A)).sum(-1)).to(torch.int32)     # [..., A] 0/1 -> bit-mask words


def run_arm(arm, model, batch, wave, inputs, rep):
    cfg = config()
    roots = batch * PER
    mask = torch.ones(batch, PER, dtype=torch.uint8).pin_memory()
    if arm == "a":
        ins = [dict(obs=expand(t["u8"]).reshape(roots, STACK * D).float().pin_memory(),
                    legal=t["legal"].reshape(roots, A).pin_memory()) for t in inputs]
        h2d = STACK * D * 4 + A * 4 + 1

        def call(k):
            t = ins[k % len(ins)]
            return reanalyze_policies(cfg, model, t["obs"], t["legal"], mask.reshape(roots), K, noise_seed=1,
                                      noise_step=k)
        for k in range(3):
            call(k)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(CALLS):
            out = call(k)
        dt = time.perf_counter() - t0
        assert abs(float(out.sum()) - roots) < 1e-6, "targets"
        rec = dict(kind="arm", arm=arm, rep=rep, batch=batch, roots_per_ticket=roots, tickets=CALLS, wave=1, depth=1,
                   window_s=round(dt, 4), host_us_per_ticket=1e6 * dt / CALLS)
    else:
        rp = ReanalyzePipeline(cfg, model, batch, K, STACK, depth=DEPTH, wave=wave)
        pipe = rp.pipe
        lw = [words(t["legal"]).pin_memory() for t in inputs]
        if arm == "b":
            ins = [(t["u8"].pin_memory(), l) for t, l in zip(inputs, lw)]
            h2d = ((K + STACK) * D + PER * (2 * 4 + 1)) / PER
        elif arm == "c":
            ins = [(expand(t["u8"]).contiguous().pin_memory(), l) for t, l in zip(inputs, lw)]
            h2d = STACK * D + 2 * 4 + 1
        else:
            ins = [(t["bits"].pin_memory(), l) for t, l in zip(inputs, lw)]
            h2d = ((K + STACK) * W * 4 + PER * (2 * 4 + 1)) / PER
        ring = DEPTH * wave + wave
        outs = [torch.empty(batch, PER, A, dtype=torch.float64).pin_memory() for _ in range(ring)]

        def submit(k):
            obs, legal = ins[k % len(ins)]
            out = outs[k % ring]
            if arm != "c":
                return rp.submit(obs, legal, mask, noise_seed=1, noise_step=k, out=out)
            # expanded stacks: the same ticket through submit_observations with positions = 1
            lg = legal.reshape(roots)
            lf = ((lg.to(dev, non_blocking=True).unsqueeze(1) >> torch.arange(A, device=dev, dtype=torch.int32)) & 1)
            noise = dirichlet_noise(roots, A, cfg.root_dirichlet_alpha, dev, 1, k) * lf.float()
            return pipe.submit_observations(cfg.root_exploration_fraction, noise, obs, lg, policy_mask=mask.reshape(roots),
                                            out_policy=out)
        for k in range(3 * DEPTH * wave):         # every slot: eager search, capture, replay
            submit(k)
        rp.drain()
        torch.cuda.synchronize()
        pipe.host_seconds, pipe.submitted = 0.0, 0
        t0 = time.perf_counter()
        for k in range(TICKETS):
            submit(k)
        rp.drain()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        assert abs(float(outs[0].sum()) - roots) < 1e-6, "targets"
        rec = dict(kind="arm", arm=arm, rep=rep, batch=batch, roots_per_ticket=roots, tickets=TICKETS, wave=wave,
                   depth=DEPTH, executor=pipe.executor, window_s=round(dt, 4),
                   host_us_per_ticket=1e6 * pipe.host_seconds / pipe.submitted)
        del rp, pipe
    n = rec["tickets"] * roots
    rec.update(positions_per_s=n / dt, sims_per_s=n * (SIMS - 1) / dt, h2d_bytes_per_position=round(h2d, 1),
               d2h_bytes_per_position=A * 8)
    emit(rec)
    torch.cuda.synchronize()
    return rec


def pack_timing(batch, wave, inputs):
    """(e) the window pack against the stack pack: one wave of `wave` tickets of batch windows (batch * PER roots) into
    fp16 x; uint8 and bit frames, pinned host and device sources; CUDA events over 200 launches."""
    lib = _lib.load()
    roots = batch * PER
    L = _lib.ObsLayout(stack=STACK, frame_dim=D, frame_stride=800, elem_bytes=2, frame_words=W, bit_offset=0)
    x = torch.empty(wave * roots, STACK * 800, dtype=torch.float16, device=dev)
    legal = torch.empty(wave * roots, A, dtype=torch.int32, device=dev)
    noise = torch.empty(wave * roots, A, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    for where in ("pinned", "device"):
        move = (lambda v: v.contiguous().pin_memory()) if where == "pinned" else (lambda v: v.contiguous().to(dev))
        for fmt in ("u8", "bits"):
            for form in ("windows", "stacks"):
                keep, table = [], []
                for t in inputs[:wave]:
                    src = t["u8"] if fmt == "u8" else t["bits"].view(batch, K + STACK, W)
                    obs = move(src if form == "windows" else expand(src))
                    lw, nz = move(words(t["legal"]).reshape(roots)), move(torch.rand(roots, A))
                    keep += [obs, lw, nz]
                    table.append(_lib.ObsTicket(obs=obs.data_ptr(), ld_obs=obs.stride(0), legal=lw.data_ptr(), ld_legal=1,
                                                noise=nz.data_ptr(), obs_format=_lib.HZ_OBS_U8 if fmt == "u8" else
                                                _lib.HZ_OBS_BITS, legal_format=_lib.HZ_LEGAL_MASK))
                tab = (_lib.ObsTicket * wave)(*table)
                if form == "windows":
                    call = lambda: _lib.check(lib.hz_obs_pack_windows(st, 0, tab, wave, wave, roots, A, ctypes.byref(L),
                                                                      PER, x.data_ptr(), legal.data_ptr(),
                                                                      noise.data_ptr()))
                else:
                    call = lambda: _lib.check(lib.hz_obs_pack(st, 0, tab, wave, wave, roots, A, ctypes.byref(L),
                                                              x.data_ptr(), legal.data_ptr(), noise.data_ptr()))
                for _ in range(20):
                    call()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                iters = 200
                e0.record()
                for _ in range(iters):
                    call()
                e1.record()
                torch.cuda.synchronize()
                us = e0.elapsed_time(e1) * 1e3 / iters
                src_bytes = sum(o.numel() * o.element_size() for o in keep)
                emit(dict(kind="pack", batch=batch, wave=wave, roots=wave * roots, source=where, fmt=fmt, form=form,
                          us_per_launch=us, source_bytes=src_bytes, source_gb_per_s=src_bytes / us / 1e3))


def report(info):
    what = {"a": "reanalyze_policies, float32 stacks, pinned host, one call at a time",
            "b": "ReanalyzePipeline, uint8 windows, pinned host",
            "c": "pipeline, uint8 stacks expanded on the host (positions = 1)",
            "d": "ReanalyzePipeline, bit-string windows, pinned host"}
    lines = ["# r05: reanalyze policy targets on the search pipeline (ReanalyzePipeline)", "",
             f"Measured on {info['device']} (nvidia-smi name, power limit, max SM clock: {info['nvidia_smi']}), "
             f"torch {info['torch']}.  Hanabi-Full, global observation, stack 4, K = 5 (6 positions per window), fp16, "
             f"50 simulations, every position kept; pipeline arms: {DEPTH} searches in flight, waves of 3 x 1536 or "
             f"1 x 4092 roots, {TICKETS} tickets per timed window, targets to pinned host memory; arm (a): {CALLS} "
             f"calls.  {REPS} repetitions (median, min-max).  Written by scripts/exp_reanalyze.py.", "",
             "| batch (roots) | arm | input | k positions/s | M simulations/s | host us / ticket | H2D B / position |",
             "|---|---|---|---|---|---|---|"]
    for batch, _ in SHAPES:
        arms = {}
        for r in RECS:
            if r["kind"] == "arm" and r["batch"] == batch:
                arms.setdefault(r["arm"], []).append(r)
        for arm in sorted(arms):
            p = [r["positions_per_s"] / 1e3 for r in arms[arm]]
            v = [r["sims_per_s"] / 1e6 for r in arms[arm]]
            h = [r["host_us_per_ticket"] for r in arms[arm]]
            lines.append(f"| {batch} ({batch * PER}) | {arm} | {what[arm]} | {statistics.median(p):.0f} | "
                         f"{statistics.median(v):.1f} ({min(v):.1f}-{max(v):.1f}) | {statistics.median(h):.0f} | "
                         f"{arms[arm][0]['h2d_bytes_per_position']} |")
        if "a" in arms and "b" in arms:
            s = statistics.median(r["sims_per_s"] for r in arms["b"]) / statistics.median(r["sims_per_s"] for r in arms["a"])
            lines.append(f"| {batch} ({batch * PER}) | b / a | speed-up | | {s:.1f}x | | |")
    lines += ["", "(e) the observation pack alone, one wave into fp16 x (CUDA events over 200 launches):", "",
              "| batch x wave (roots) | source | frames | form | us / launch | source bytes | source GB/s |",
              "|---|---|---|---|---|---|---|"]
    for r in RECS:
        if r["kind"] == "pack":
            lines.append(f"| {r['batch']} x {r['wave']} ({r['roots']}) | {r['source']} | {r['fmt']} | {r['form']} | "
                         f"{r['us_per_launch']:.1f} | {r['source_bytes']} | {r['source_gb_per_s']:.1f} |")
    with open(os.path.join(OUT, "r05_reanalyze.md"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines), flush=True)


if __name__ == "__main__":
    try:
        info = card()
        emit(dict(kind="setup", **info, cuda_device_max_connections=os.environ["CUDA_DEVICE_MAX_CONNECTIONS"]))
        torch.manual_seed(0)
        model = MuZeroNetFull(D * STACK, A).randomize_heads(seed=0).to(dev).eval()
        for batch, wave in SHAPES:
            inputs = [windows(batch, 1000 * i) for i in range(INPUTS)]
            for rep in range(REPS):
                for arm in ("a", "b", "c", "d"):
                    run_arm(arm, model, batch, wave, inputs, rep)
            pack_timing(batch, wave, inputs)
        report(info)
    except Exception:
        traceback.print_exc()
        sys.exit(1)
