"""Experiment: reanalyze tickets read from an episode store in device memory (ReanalyzePipeline.submit_episodes) against
tickets of frame windows (ReanalyzePipeline.submit).  Hanabi-Full, global observation, stack 4, K = 5 (6 positions per
window), fp16 (torch_amp), 50 simulations, 8 searches in flight, batches of 256 and 682 windows per ticket (waves of
3 x 1536 and 1 x 4092 roots), the same real-play windows as scripts/exp_reanalyze.py:
  (store)  submit_episodes: each window is a stored episode of T = K + 1 moves, sampled at start 0; the host hands in
           16 bytes per sample
  (b)      submit of uint8 windows [batch, K + 4, 785] + legal bit-mask words + mask from pinned host memory (r05 arm b)
  (dev)    submit of the same windows, words and mask already in device memory
Every arm writes its targets to pinned host memory and computes the same targets (checked).  Rates count every
position and 49 simulations per position; the timed window submits TICKETS tickets and ends with drain() + a
synchronise.  Host us per ticket = the pipeline's host_seconds / submitted.  H2D bytes per position are computed from
the shapes each arm hands in.  Then the pack alone per arm (hz_obs_pack_episodes from the store, hz_obs_pack_windows
from pinned and from device memory), one wave into fp16 x, CUDA events over 200 launches.  Writes
OUT/r06_episode_store.jsonl and OUT/r06_episode_store.md; the card and its power limit are read in the same run.
Env: OUT (default /tmp/reanalyze_store), TICKETS (150), REPS (2)."""
import os
import sys

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ctypes
import json
import statistics
import time
import traceback

import numpy as np
import torch

from exp_reanalyze import A, D, K, PER, SIMS, STACK, card, config, windows, words
from hanabizero_b200 import _lib
from hanabizero_b200.model import MuZeroNetFull
from hanabizero_b200.reanalyze import ReanalyzePipeline
from hanabizero_b200.trajectory import EpisodeStore

OUT = os.environ.get("OUT", "/tmp/reanalyze_store")
TICKETS = int(os.environ.get("TICKETS", "150"))
REPS = int(os.environ.get("REPS", "2"))
DEPTH = 8
SHAPES = [(256, 3), (682, 1)]
INPUTS = 4
dev = torch.device("cuda")
os.makedirs(OUT, exist_ok=True)
RECS = []


def emit(rec):
    print(json.dumps(rec), flush=True)
    RECS.append(rec)
    with open(os.path.join(OUT, "r06_episode_store.jsonl"), "a") as f:
        f.write(json.dumps(rec) + "\n")


def fill_store(inputs, batch):
    """Every window as an episode of K + 1 moves (its first STACK frames stand for the stack copies, then its frames and
    one more, the legal rows of its positions and one more): sample (id, 0) reads exactly the window, its legal rows
    and an all-kept mask."""
    store = EpisodeStore(INPUTS * batch * (STACK + PER) + 16, D, A, STACK)
    ids = []
    for t in inputs:
        o = torch.cat([t["u8"], t["u8"][:, -1:]], 1).numpy()
        la = torch.cat([t["legal"], t["legal"][:, -1:]], 1).numpy()
        ids.append(store.add([dict(o=o[b], la=la[b]) for b in range(batch)]))
    torch.cuda.synchronize()
    return store, ids


def run_arm(arm, model, batch, wave, inputs, store, ids, rep):
    cfg = config()
    roots = batch * PER
    rp = ReanalyzePipeline(cfg, model, batch, K, STACK, depth=DEPTH, wave=wave)
    pipe = rp.pipe
    mask = torch.ones(batch, PER, dtype=torch.uint8)
    starts = np.zeros(batch, np.int64)
    if arm == "b":
        ins = [(t["u8"].pin_memory(), words(t["legal"]).pin_memory(), mask.pin_memory()) for t in inputs]
        h2d = ((K + STACK) * D + PER * (4 + 1)) / PER
    elif arm == "dev":
        ins = [(t["u8"].to(dev), words(t["legal"]).to(dev), mask.to(dev)) for t in inputs]
        h2d = 0.0
    else:
        h2d = 16 / PER
    ring = DEPTH * wave + wave
    outs = [torch.empty(batch, PER, A, dtype=torch.float64).pin_memory() for _ in range(ring)]

    def submit(k):
        out = outs[k % ring]
        if arm == "store":
            return rp.submit_episodes(store, ids[k % len(ids)], starts, noise_seed=1, noise_step=k, out=out)
        obs, legal, m = ins[k % len(ins)]
        return rp.submit(obs, legal, m, noise_seed=1, noise_step=k, out=out)

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
    n = TICKETS * roots
    rec = dict(kind="arm", arm=arm, rep=rep, batch=batch, roots_per_ticket=roots, tickets=TICKETS, wave=wave,
               depth=DEPTH, executor=pipe.executor, window_s=round(dt, 4),
               host_us_per_ticket=1e6 * pipe.host_seconds / pipe.submitted, positions_per_s=n / dt,
               sims_per_s=n * (SIMS - 1) / dt, h2d_bytes_per_position=round(h2d, 1), d2h_bytes_per_position=A * 8)
    emit(rec)
    last = [o.clone() for o in outs[:2]]
    del rp, pipe
    torch.cuda.synchronize()
    return last


def pack_timing(batch, wave, inputs, store, ids):
    """The pack alone, one wave of `wave` tickets of batch windows into fp16 x: from the store (hz_obs_pack_episodes),
    and from uint8 windows in pinned and in device memory (hz_obs_pack_windows); CUDA events over 200 launches."""
    lib = _lib.load()
    roots = batch * PER
    L = _lib.ObsLayout(stack=STACK, frame_dim=D, frame_stride=800, elem_bytes=2, frame_words=25, bit_offset=0)
    x = torch.empty(wave * roots, STACK * 800, dtype=torch.float16, device=dev)
    legal = torch.empty(wave * roots, A, dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    outs = {}
    for src in ("store", "pinned", "device"):
        keep, table = [], []
        for t, i in zip(inputs[:wave], ids[:wave]):
            nz = torch.rand(roots, A, device=dev)
            if src == "store":
                smp = torch.from_numpy(store.samples(i, np.zeros(batch, np.int64), PER)).to(dev)
                m = torch.empty(roots, dtype=torch.uint8, device=dev)
                keep += [smp, m, nz]
                table.append(_lib.EpisodeTicket(frames=store.frames.data_ptr(), ld_frames=D,
                                                legal=store.legal.data_ptr(), samples=smp.data_ptr(),
                                                noise=nz.data_ptr(), mask=m.data_ptr()))
            else:
                move = (lambda v: v.contiguous().pin_memory()) if src == "pinned" else (lambda v: v.contiguous().to(dev))
                obs, lw = move(t["u8"]), move(words(t["legal"]).reshape(roots))
                keep += [obs, lw, nz]
                table.append(_lib.ObsTicket(obs=obs.data_ptr(), ld_obs=obs.stride(0), legal=lw.data_ptr(), ld_legal=1,
                                            noise=nz.data_ptr(), obs_format=_lib.HZ_OBS_U8,
                                            legal_format=_lib.HZ_LEGAL_MASK))
        if src == "store":
            tab = (_lib.EpisodeTicket * wave)(*table)
            call = lambda: _lib.check(lib.hz_obs_pack_episodes(st, 0, tab, wave, wave, roots, A, ctypes.byref(L), PER,
                                                               x.data_ptr(), legal.data_ptr(), None))
        else:
            tab = (_lib.ObsTicket * wave)(*table)
            call = lambda: _lib.check(lib.hz_obs_pack_windows(st, 0, tab, wave, wave, roots, A, ctypes.byref(L), PER,
                                                              x.data_ptr(), legal.data_ptr(), None))
        for _ in range(20):
            call()
        torch.cuda.synchronize()
        outs[src] = (x.clone(), legal.clone())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters = 200
        e0.record()
        for _ in range(iters):
            call()
        e1.record()
        torch.cuda.synchronize()
        emit(dict(kind="pack", batch=batch, wave=wave, roots=wave * roots, source=src,
                  us_per_launch=e0.elapsed_time(e1) * 1e3 / iters))
    for src in ("pinned", "device"):
        assert torch.equal(outs["store"][0].view(torch.int16), outs[src][0].view(torch.int16)), src
        assert torch.equal(outs["store"][1], outs[src][1]), src


def report(info):
    what = {"store": "submit_episodes: (id, start) into the device store",
            "b": "submit: uint8 windows, pinned host (r05 arm b)",
            "dev": "submit: uint8 windows already in device memory"}
    lines = ["# r06: reanalyze tickets from an episode store in device memory", "",
             f"Measured on {info['device']} (nvidia-smi name, power limit, max SM clock: {info['nvidia_smi']}), "
             f"torch {info['torch']}.  Hanabi-Full, global observation, stack 4, K = 5 (6 positions per window), fp16, "
             f"50 simulations, every position kept; {DEPTH} searches in flight, waves of 3 x 1536 or 1 x 4092 roots, "
             f"{TICKETS} tickets per timed window, targets to pinned host memory.  {REPS} repetitions (median, "
             f"min-max).  Written by scripts/exp_reanalyze_store.py.", "",
             "| batch (roots) | arm | input | k positions/s | M simulations/s | host us / ticket | H2D B / position |",
             "|---|---|---|---|---|---|---|"]
    for batch, _ in SHAPES:
        arms = {}
        for r in RECS:
            if r["kind"] == "arm" and r["batch"] == batch:
                arms.setdefault(r["arm"], []).append(r)
        for arm in ("store", "b", "dev"):
            if arm not in arms:
                continue
            p = [r["positions_per_s"] / 1e3 for r in arms[arm]]
            v = [r["sims_per_s"] / 1e6 for r in arms[arm]]
            h = [r["host_us_per_ticket"] for r in arms[arm]]
            lines.append(f"| {batch} ({batch * PER}) | {arm} | {what[arm]} | {statistics.median(p):.0f} | "
                         f"{statistics.median(v):.1f} ({min(v):.1f}-{max(v):.1f}) | {statistics.median(h):.0f} | "
                         f"{arms[arm][0]['h2d_bytes_per_position']} |")
    lines += ["", "The pack alone, one wave into fp16 x (CUDA events over 200 launches; the three give identical x and "
              "legal rows):", "", "| batch x wave (roots) | source | us / launch |", "|---|---|---|"]
    for r in RECS:
        if r["kind"] == "pack":
            lines.append(f"| {r['batch']} x {r['wave']} ({r['roots']}) | {r['source']} | {r['us_per_launch']:.1f} |")
    with open(os.path.join(OUT, "r06_episode_store.md"), "w") as f:
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
            store, ids = fill_store(inputs, batch)
            for rep in range(REPS):
                res = {arm: run_arm(arm, model, batch, wave, inputs, store, ids, rep) for arm in ("store", "b", "dev")}
                for arm in ("b", "dev"):       # the same tickets in the same ring positions: the same targets
                    assert all(torch.equal(x.view(torch.int64), y.view(torch.int64))
                               for x, y in zip(res["store"], res[arm])), arm
            pack_timing(batch, wave, inputs, store, ids)
        report(info)
    except Exception:
        traceback.print_exc()
        sys.exit(1)
