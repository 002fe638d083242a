"""Experiment: searches that start from observations (SearchPipeline.submit_observations) against today's ways of
handing a search its roots.  Hanabi-Full, global observation, stack 4, fp16 (torch_amp), 50 simulations, one GPU,
tickets of 512 roots in waves of 8 (4096 trees per search), 20 searches in flight:
  (a) observation tickets as packed bits (+ the legal mask word) from pinned host memory
  (b) observation tickets as float32 frames (+ float legal mask) from pinned host memory
  (c) the caller runs model.initial_inference_device on the float frames (copied from pinned host memory), then
      submit(hidden) — what a host-driven actor has to do without (a) / (b)
  (d) hidden-state tickets already on the device (noise, reward, logits, legal, fp16 hidden): the existing upper bound
Rates count 512 * 49 simulations per ticket; the timed window submits TICKETS tickets and ends with drain() + a
synchronise.  Host us per ticket = SearchPipeline.host_seconds / submitted (for (c) the caller's own host time around
the module call is added).  H2D bytes per root are computed from the shapes the arm hands in.  Then hz_obs_pack alone,
timed with CUDA events over many launches, and a closed host-driven actor loop (EnvPipeline(fmt="bits") groups -> host
frame stack of bit rows -> submit_observations -> host arg-max -> step) next to SelfPlayPool's device-resident moves at
the same game count.  Writes OUT/r04_obs_search.jsonl and OUT/r04_obs_search.md; the card and its power limit are read
in the same run.  Env: OUT (default /tmp/obs_search), TICKETS (2400), REPS (3), MOVES (40)."""
import os
import sys

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before CUDA starts: 20 searches in flight need > 8 queues
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
from hanabizero_b200.hanabi_env import EnvPipeline, HanabiVecEnv
from hanabizero_b200.mcts import MCTS, SearchConfig, SearchPipeline
from hanabizero_b200.model import MuZeroNetFull
from hanabizero_b200.selfplay import SelfPlayEngine, SelfPlayPool

OUT = os.environ.get("OUT", "/tmp/obs_search")
TICKETS = int(os.environ.get("TICKETS", "2400"))
REPS = int(os.environ.get("REPS", "3"))
MOVES = int(os.environ.get("MOVES", "40"))
N, G, DEPTH, S, STACK, A = 512, 8, 20, 50, 4, 20
dev = torch.device("cuda")
os.makedirs(OUT, exist_ok=True)
RECS = []


def emit(rec):
    print(json.dumps(rec), flush=True)
    RECS.append(rec)
    with open(os.path.join(OUT, "r04_obs_search.jsonl"), "a") as f:
        f.write(json.dumps(rec) + "\n")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    return dict(device=torch.cuda.get_device_name(0), nvidia_smi=line, torch=torch.__version__)


def positions(count):
    """`count` tickets of real Hanabi-Full positions (reset + 10 random moves): frames (the observation repeated over
    the stack) as float32 and as packed bits, legal masks as float, int32 and bit-mask words, noise."""
    env = HanabiVecEnv(N * count, "Hanabi-Full", np.arange(N * count))
    g, _, legal = env.reset_all()
    gen = torch.Generator(device=dev).manual_seed(3)
    for _ in range(10):
        g, _, legal, _, _, _ = env.step_all(torch.multinomial(legal, 1, generator=gen).view(-1).int(), auto_reset=True)
    env.check()
    rows = env.step_bits(None).cpu()                     # [n, W + 4]: observation words, legal mask word, ...
    W = env.bits_words - 4
    rng = np.random.default_rng(7)
    out = []
    for k in range(count):
        r = slice(k * N, (k + 1) * N)
        words = rows[r, :W]
        out.append(dict(bits=words.unsqueeze(1).repeat(1, STACK, 1).contiguous(), meta=rows[r, W:].contiguous(),
                        f32=g[r].repeat(1, STACK).cpu(), legal_f=legal[r].cpu(), legal_i=legal[r].int().cpu(),
                        noise=torch.from_numpy(rng.dirichlet([0.3] * A, N).astype(np.float32))))
    return out


def pinned(t):
    return {k: v.pin_memory() for k, v in t.items()}


def run_arm(arm, model, tickets, rep):
    cfg = SearchConfig(num_simulations=S, amp_type="torch_amp")
    obs_arm = arm in ("a", "b")
    pipe = SearchPipeline(MCTS(cfg), model, N, A, depth=DEPTH, wave=G, stack=STACK if obs_arm else None)
    outs = [(torch.empty(N, A, dtype=torch.int32).pin_memory(), torch.empty(N).pin_memory()) for _ in range(2 * G)]
    extra_host = [0.0]
    if arm == "a":
        ins = [pinned(dict(obs=t["bits"], meta=t["meta"], noise=t["noise"])) for t in tickets]
        h2d = STACK * ins[0]["obs"].shape[2] * 4 + 4 + A * 4

        def submit(t, o):
            pipe.submit_observations(0.25, t["noise"], t["obs"], t["meta"][:, 0], o[0], o[1])
    elif arm == "b":
        ins = [pinned(dict(obs=t["f32"], legal=t["legal_f"], noise=t["noise"])) for t in tickets]
        h2d = STACK * 785 * 4 + 2 * A * 4

        def submit(t, o):
            pipe.submit_observations(0.25, t["noise"], t["obs"], t["legal"], o[0], o[1])
    elif arm == "c":
        ins = [pinned(dict(obs=t["f32"], legal=t["legal_i"], noise=t["noise"])) for t in tickets]
        zeros = torch.zeros(N, device=dev)
        h2d = STACK * 785 * 4 + 2 * A * 4

        def submit(t, o):
            t0 = time.perf_counter()
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
                _, logits, hidden = model.initial_inference_device(t["obs"].to(dev, non_blocking=True))
            logits = logits.float()
            extra_host[0] += time.perf_counter() - t0
            pipe.submit(0.25, t["noise"], zeros, logits, t["legal"], hidden, o[0], o[1])
    else:
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            ins = []
            for t in tickets:
                _, logits, hidden = model.initial_inference_device(t["f32"].to(dev))
                ins.append(dict(noise=t["noise"].to(dev), reward=torch.zeros(N, device=dev),
                                logits=logits.float().contiguous(), legal=t["legal_i"].to(dev), hidden=hidden.contiguous()))
        h2d = 0

        def submit(t, o):
            pipe.submit(0.25, t["noise"], t["reward"], t["logits"], t["legal"], t["hidden"], o[0], o[1])
    for k in range(3 * DEPTH * G):              # every slot: eager search, capture, replay
        submit(ins[k % len(ins)], outs[k % len(outs)])
    pipe.drain()
    torch.cuda.synchronize()
    pipe.host_seconds, pipe.submitted, extra_host[0] = 0.0, 0, 0.0
    t0 = time.perf_counter()
    for k in range(TICKETS):
        submit(ins[k % len(ins)], outs[k % len(outs)])
    pipe.drain()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    assert int(outs[0][0].sum()) == N * (S - 1), "search result"
    rec = dict(kind="arm", arm=arm, rep=rep, tickets=TICKETS, roots_per_ticket=N, wave=G, depth=DEPTH,
               executor=pipe.executor, window_s=round(dt, 4), sims_per_s=TICKETS * N * (S - 1) / dt,
               host_us_per_ticket=1e6 * (pipe.host_seconds + extra_host[0]) / pipe.submitted, h2d_bytes_per_root=h2d)
    emit(rec)
    del pipe
    torch.cuda.synchronize()
    return rec


def pack_timing(tickets):
    """hz_obs_pack alone: one wave of 8 tickets x 512 roots into fp16 x, CUDA events over ITER launches."""
    lib = _lib.load()
    W = tickets[0]["bits"].shape[2]
    L = _lib.ObsLayout(stack=STACK, frame_dim=785, frame_stride=800, elem_bytes=2, frame_words=W, bit_offset=0)
    x = torch.empty(G * N, STACK * 800, dtype=torch.float16, device=dev)
    legal = torch.empty(G * N, A, dtype=torch.int32, device=dev)
    noise = torch.empty(G * N, A, device=dev)
    cases = []
    for where in ("pinned", "device"):
        for fmt in ("bits", "f32"):
            keep, table = [], []
            for t in tickets[:G]:
                move = (lambda v: v.pin_memory()) if where == "pinned" else (lambda v: v.to(dev))
                obs = move(t["bits"] if fmt == "bits" else t["f32"])
                meta, leg, nz = move(t["meta"]), move(t["legal_f"]), move(t["noise"])
                keep += [obs, meta, leg, nz]
                if fmt == "bits":
                    table.append(_lib.ObsTicket(obs=obs.data_ptr(), ld_obs=obs.stride(0), legal=meta.data_ptr(), ld_legal=4,
                                                noise=nz.data_ptr(), obs_format=_lib.HZ_OBS_BITS,
                                                legal_format=_lib.HZ_LEGAL_MASK))
                else:
                    table.append(_lib.ObsTicket(obs=obs.data_ptr(), ld_obs=obs.stride(0), legal=leg.data_ptr(), ld_legal=A,
                                                noise=nz.data_ptr(), obs_format=_lib.HZ_OBS_F32,
                                                legal_format=_lib.HZ_LEGAL_F32))
            src = N * G * ((STACK * W * 4 + 4) if fmt == "bits" else (STACK * 785 * 4 + A * 4)) + N * G * A * 4
            cases.append((where, fmt, (_lib.ObsTicket * G)(*table), keep, src))
    st = torch.cuda.current_stream().cuda_stream
    written = x.numel() * 2 + legal.numel() * 4 + noise.numel() * 4
    for where, fmt, tab, keep, src in cases:
        call = lambda: _lib.check(lib.hz_obs_pack(st, 0, tab, G, G, N, A, ctypes.byref(L), x.data_ptr(), legal.data_ptr(),
                                                  noise.data_ptr()))
        for _ in range(20):
            call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters = 500
        e0.record()
        for _ in range(iters):
            call()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / iters
        emit(dict(kind="pack", source=where, fmt=fmt, roots=G * N, us_per_launch=us, source_bytes=src,
                  written_bytes=written, read_gb_per_s=src / us / 1e3, total_gb_per_s=(src + written) / us / 1e3))


def actor_loop(model, groups, games):
    """Closed host-driven loop over `groups` EnvPipeline groups of `games` games: per move and group, wait for the
    group's rows, push its packed frame into a host stack of bit rows, submit_observations (bit frames + the meta rows'
    legal mask word), then per group wait for the search, arg-max on the host, step.  -> moves (games x steps) / s."""
    envs = [HanabiVecEnv(games, "Hanabi-Full", np.arange(games) + 7919 * g) for g in range(groups)]
    for e in envs:
        e.reset_all(observe=False)
    W = envs[0].bits_words - 4
    pipe = SearchPipeline(MCTS(SearchConfig(num_simulations=S, amp_type="torch_amp")), model, games, A, depth=groups,
                          stack=STACK)
    ep = EnvPipeline(envs, fmt="bits")
    stacks = [torch.zeros(games, STACK, W, dtype=torch.int32).pin_memory() for _ in range(groups)]
    visits = [torch.zeros(games, A, dtype=torch.int32).pin_memory() for _ in range(groups)]
    for g in range(groups):
        ep.observe_now(g)
    first = [True] * groups

    def move():
        tids = []
        for g in range(groups):
            words, meta = ep.wait(g)
            st = stacks[g]
            st[:, :-1] = st[:, 1:].clone()
            st[:, -1] = words
            new = torch.ones(games, dtype=torch.bool) if first[g] else meta[:, 2] != 0
            first[g] = False
            st[new] = words[new].unsqueeze(1).expand(-1, STACK, -1)
            tids.append(pipe.submit_observations(0.0, None, st, meta[:, 0], visits[g]))
        for g in range(groups):
            pipe.wait(tids[g])
            ep.step(g, visits[g].argmax(1).int())

    for _ in range(5):
        move()
    ep.drain()
    torch.cuda.synchronize()
    pipe.host_seconds, pipe.submitted = 0.0, 0
    t0 = time.perf_counter()
    for _ in range(MOVES):
        move()
    ep.drain()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    for e in envs:
        e.check()
    return dict(kind="actor_loop", groups=groups, games_per_group=games, moves=MOVES, window_s=round(dt, 4),
                moves_per_s=groups * games * MOVES / dt, host_us_per_ticket=1e6 * pipe.host_seconds / pipe.submitted)


def selfplay_pool(model, groups, games):
    cfg = SearchConfig(num_simulations=S, amp_type="torch_amp")
    pool = SelfPlayPool([SelfPlayEngine(games, "Hanabi-Full", model, cfg, seeds=np.arange(games) + 7919 * g)
                         for g in range(groups)])
    pool.reset()
    for _ in range(5):
        pool.step(deterministic=True, noise=False)
    pool.synchronize()
    t0 = time.perf_counter()
    for _ in range(MOVES):
        pool.step(deterministic=True, noise=False)
    pool.synchronize()
    dt = time.perf_counter() - t0
    return dict(kind="selfplay_pool", groups=groups, games_per_group=games, moves=MOVES, window_s=round(dt, 4),
                moves_per_s=groups * games * MOVES / dt)


def report(info):
    arms = {}
    for r in RECS:
        if r["kind"] == "arm":
            arms.setdefault(r["arm"], []).append(r)
    what = {"a": "observation tickets, packed bits, pinned host", "b": "observation tickets, float32, pinned host",
            "c": "caller's initial_inference_device on float frames, then submit(hidden)",
            "d": "hidden-state tickets on the device (upper bound)"}
    lines = ["# r04: searches that start from observations (SearchPipeline.submit_observations)", "",
             f"Measured on {info['device']} (nvidia-smi name, power limit, max SM clock: {info['nvidia_smi']}), "
             f"torch {info['torch']}.  Hanabi-Full, global observation, stack 4, fp16, 50 simulations; tickets of "
             f"{N} roots in waves of {G}, {DEPTH} searches in flight; {TICKETS} tickets per timed window, "
             f"{REPS} repetitions (median, min-max).  Written by scripts/exp_obs_search.py.", "",
             "| arm | input | M simulations/s | host us / ticket | H2D bytes / root |", "|---|---|---|---|---|"]
    for arm in sorted(arms):
        v = [r["sims_per_s"] / 1e6 for r in arms[arm]]
        h = [r["host_us_per_ticket"] for r in arms[arm]]
        lines.append(f"| {arm} | {what[arm]} | {statistics.median(v):.1f} ({min(v):.1f}-{max(v):.1f}) | "
                     f"{statistics.median(h):.1f} | {arms[arm][0]['h2d_bytes_per_root']} |")
    lines += ["", "hz_obs_pack alone (one wave: 8 tickets x 512 roots -> fp16 x [4096, 3200], legal, noise; CUDA events "
              "over 500 launches):", "", "| source | format | us / launch | source GB/s | read + written GB/s |",
              "|---|---|---|---|---|"]
    for r in RECS:
        if r["kind"] == "pack":
            lines.append(f"| {r['source']} | {r['fmt']} | {r['us_per_launch']:.1f} | {r['read_gb_per_s']:.1f} | "
                         f"{r['total_gb_per_s']:.1f} |")
    lines += ["", "Closed loop (Hanabi-Full, arg-max actions, no noise):", "",
              "| loop | groups x games | moves / s | host us / ticket |", "|---|---|---|---|"]
    for r in RECS:
        if r["kind"] == "actor_loop":
            lines.append(f"| host-driven: EnvPipeline bits -> submit_observations -> host arg-max | {r['groups']} x "
                         f"{r['games_per_group']} | {r['moves_per_s']:.0f} | {r['host_us_per_ticket']:.1f} |")
        elif r["kind"] == "selfplay_pool":
            lines.append(f"| device-resident: SelfPlayPool | {r['groups']} x {r['games_per_group']} | "
                         f"{r['moves_per_s']:.0f} | - |")
    with open(os.path.join(OUT, "r04_obs_search.md"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines), flush=True)


if __name__ == "__main__":
    try:
        info = card()
        emit(dict(kind="setup", **info, cuda_device_max_connections=os.environ["CUDA_DEVICE_MAX_CONNECTIONS"]))
        torch.manual_seed(0)
        model = MuZeroNetFull(785 * STACK, A).randomize_heads(seed=0).to(dev).eval()
        tickets = positions(G)
        for rep in range(REPS):
            for arm in ("a", "b", "c", "d"):
                run_arm(arm, model, tickets, rep)
        pack_timing(tickets)
        emit(actor_loop(model, 8, N))
        emit(selfplay_pool(model, 8, N))
        report(info)
    except Exception:
        traceback.print_exc()
        sys.exit(1)
