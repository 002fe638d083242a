"""Experiment: what recording costs a self-play pool.  Hanabi-Full, global observation, stack 4, fp16 (torch_amp),
50 simulations, sampled moves with root noise (SelfPlayPool.step() defaults), random-init network with re-drawn heads.
Two pool shapes: 7 engines x 4096 games (bench.py's self-play setting) and 20 engines x 512 games; the process runs
with CUDA_DEVICE_MAX_CONNECTIONS=32 (set before CUDA starts, as bench.py does), which 20 streams need.  Three arms:
  off     SelfPlayEngine(record=False): the unrecorded fast path (byte frame ring, InitialPlan, auto-reset in the env)
  legacy  SelfPlayEngine(record=True): float frame stack, the module's root inference, step without auto-reset, masked
          reset, second observe, hz_traj_append + hz_traj_begin
  ring    SelfPlayEngine(record="ring"): the fast path plus the terminal-row env step and one hz_traj_record_u8 launch
Timed window: SEGMENTS segments of FLUSH moves; a segment is FLUSH x pool.step() and pool.synchronize(), then (recording
arms) pool.flush().  moves/s with flushes = games x moves / (segments + flushes); without = games x moves / segments;
host ms per flush = host clock around pool.flush() (it synchronises every engine's stream and copies the episodes).  The
unrecorded arm runs the same segments with nothing after them.  Banks and cadence: a Hanabi-Full episode lasts at least
three moves (three lost lives), so a game finishes at most 3 episodes in 8 moves (at moves 1, 4, 7) and needs a fourth
bank for the episode it then begins: BANKS = 4, FLUSH = 8, and max_len = 128 holds any Hanabi-Full episode (< 100
moves).  Every flush checks the sticky overflow flag, so a run that overflowed raises instead of reporting.  The arms
run alternately, REPS times.  Writes OUT/r05_selfplay_record.{jsonl,md}; the card and its power limit are read in the
same run.  Env: OUT (default /tmp/selfplay_record), REPS (2), SEGMENTS (12), FLUSH (8), BANKS (4)."""
import os
import sys

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before CUDA starts: 20 engines need > 8 queues
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import json
import statistics
import subprocess
import time
import traceback

import numpy as np
import torch

from hanabizero_b200.mcts import SearchConfig
from hanabizero_b200.model import MuZeroNetFull
from hanabizero_b200.selfplay import SelfPlayEngine, SelfPlayPool

OUT = os.environ.get("OUT", "/tmp/selfplay_record")
REPS = int(os.environ.get("REPS", "2"))
SEGMENTS = int(os.environ.get("SEGMENTS", "12"))
FLUSH = int(os.environ.get("FLUSH", "8"))
BANKS = int(os.environ.get("BANKS", "4"))
MAX_LEN, S, STACK, A, D = 128, 50, 4, 20, 785
SHAPES = [(7, 4096), (20, 512)]
ARMS = {"off": False, "legacy": True, "ring": "ring"}
dev = torch.device("cuda")
os.makedirs(OUT, exist_ok=True)
RECS = []


def emit(rec):
    print(json.dumps(rec), flush=True)
    RECS.append(rec)
    with open(os.path.join(OUT, "r05_selfplay_record.jsonl"), "a") as f:
        f.write(json.dumps(rec) + "\n")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return dict(device=torch.cuda.get_device_name(0), nvidia_smi=line, torch=torch.__version__)


def run(model, arm, E, N, rep):
    cfg = SearchConfig(num_simulations=S, amp_type="torch_amp")
    engines = [SelfPlayEngine(N, "Hanabi-Full", model, cfg, seeds=np.arange(N) + 7 * N * (e + 1), mdp="global",
                              stack=STACK, device=dev, record=ARMS[arm], max_episode_len=MAX_LEN, record_banks=BANKS,
                              game_offset=e * N) for e in range(E)]
    pool = SelfPlayPool(engines)
    recording = arm != "off"
    pool.reset()
    for _ in range(3):                  # eager search, capture, replay
        pool.step()
    pool.synchronize()
    if recording:
        pool.flush()
    seg, fl, episodes, steps = 0.0, [], 0, 0
    for _ in range(SEGMENTS):
        t0 = time.perf_counter()
        for _ in range(FLUSH):
            pool.step()
        pool.synchronize()
        t1 = time.perf_counter()
        seg += t1 - t0
        if recording:
            eps = pool.flush()
            fl.append(time.perf_counter() - t1)
            episodes += sum(len(x) for x in eps)
            steps += sum(len(ep["a"]) for x in eps for ep in x)
    for eng in engines:
        eng.env.check()
    moves = E * N * FLUSH * SEGMENTS
    rec = dict(kind="arm", arm=arm, engines=E, games=N, rep=rep, moves=moves, segment_s=round(seg, 4),
               flush_s=round(sum(fl), 4), moves_per_s_with_flush=moves / (seg + sum(fl)), moves_per_s_without_flush=moves / seg,
               host_ms_per_flush=1e3 * statistics.mean(fl) if fl else 0.0, flushes=len(fl), episodes=episodes,
               mean_episode_moves=steps / episodes if episodes else 0.0)
    emit(rec)
    del pool, engines
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return rec


def report(info):
    lines = ["# r05: recorded self-play on the byte frame ring (SelfPlayEngine(record=\"ring\"))", "",
             f"Measured on {info['device']} (nvidia-smi name, power limit, max SM clock: {info['nvidia_smi']}), "
             f"torch {info['torch']}, CUDA_DEVICE_MAX_CONNECTIONS={os.environ['CUDA_DEVICE_MAX_CONNECTIONS']}.  "
             f"Hanabi-Full, global observation, stack {STACK}, fp16, {S} simulations, sampled moves with root noise, "
             f"random-init network.  {BANKS} record banks per game, max_len {MAX_LEN}, pool.flush() every {FLUSH} moves, "
             f"{SEGMENTS} flushes per timed window; arms run alternately, {REPS} times (both values shown, median "
             "first).  Written by scripts/exp_selfplay_record.py.", "",
             "| engines x games | arm | M moves/s with flushes | M moves/s without flushes | vs off (without flushes) | "
             "host ms / flush | episodes / flush | moves / episode |", "|---|---|---|---|---|---|---|---|"]
    what = {"off": "off (record=False)", "legacy": "legacy (record=True)", "ring": "ring (record=\"ring\")"}
    for E, N in SHAPES:
        by = {a: [r for r in RECS if r["kind"] == "arm" and r["arm"] == a and r["engines"] == E] for a in ARMS}
        base = statistics.median(r["moves_per_s_without_flush"] for r in by["off"]) if by["off"] else None
        for a in ARMS:
            rs = by[a]
            if not rs:
                continue
            w = [r["moves_per_s_with_flush"] / 1e6 for r in rs]
            wo = [r["moves_per_s_without_flush"] / 1e6 for r in rs]
            fmt = lambda v: f"{statistics.median(v):.2f} ({' / '.join(f'{x:.2f}' for x in v)})"
            rel = f"{100 * statistics.median(wo) * 1e6 / base:.1f} %" if base else "-"
            fl = statistics.median(r["host_ms_per_flush"] for r in rs)
            eps = statistics.median(r["episodes"] / max(r["flushes"], 1) for r in rs)
            ml = statistics.median(r["mean_episode_moves"] for r in rs)
            lines.append(f"| {E} x {N} | {what[a]} | {fmt(w)} | {fmt(wo)} | {rel} | "
                         f"{fl:.1f} | {eps:.0f} | {ml:.1f} |" if a != "off" else
                         f"| {E} x {N} | {what[a]} | {fmt(w)} | {fmt(wo)} | 100 % | - | - | - |")
    with open(os.path.join(OUT, "r05_selfplay_record.md"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines), flush=True)


if __name__ == "__main__":
    try:
        info = card()
        emit(dict(kind="setup", **info, cuda_device_max_connections=os.environ["CUDA_DEVICE_MAX_CONNECTIONS"],
                  banks=BANKS, flush_every=FLUSH, segments=SEGMENTS, max_len=MAX_LEN))
        torch.manual_seed(0)
        model = MuZeroNetFull(D * STACK, A).randomize_heads(seed=0).to(dev).eval()
        for rep in range(REPS):
            for E, N in SHAPES:
                for arm in ARMS:
                    run(model, arm, E, N, rep)
        report(info)
    except Exception:
        traceback.print_exc()
        sys.exit(1)
