"""Experiment: search waves.  G tickets of n trees searched as one batch of G*n trees in one SearchPipeline slot
(wave=G) against today's configuration of one search per ticket (wave=1, depth 20), on one GPU, in the same process.
  (a) wave=1, depth=20        (b) wave=4096//n, depth=8
Hanabi-Full fp16 (torch_amp), 50 simulations, device-resident inputs, tickets of n = 512, 1024, 2048, (a) and (b)
alternated REPS times; then pinned-host inputs and outputs at n = 512 and Hanabi-Small at n = 512.  A rate counts
n * (num_simulations - 1) simulations per ticket, as bench.py does; the timed window submits TREES trees in all and
ends with drain() + synchronize.  Host us per ticket = SearchPipeline.host_seconds / submitted over the window.
Last, torch.profiler traces of (a) and (b) at n = 512 go to OUT/wave_{a,b}512.pt.trace.json, kernel tables beside them.
One JSON line per run is appended to OUT/wave.jsonl.  Env: OUT (default /tmp/wave), REPS (3), TREES (4194304: windows of 1-2 s)."""
import os
import sys

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before CUDA starts: depth-20 pipelines need > 8 queues
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import json
import statistics
import time
import traceback

import numpy as np
import torch

from hanabizero_b200.mcts import MCTS, SearchConfig, SearchPipeline
from hanabizero_b200.model import MuZeroNet, MuZeroNetFull

OUT = os.environ.get("OUT", "/tmp/wave")
REPS = int(os.environ.get("REPS", "3"))
TREES = int(os.environ.get("TREES", str(4096 * 1024)))
S = 50
dev = torch.device("cuda")
os.makedirs(OUT, exist_ok=True)


def make_model(net):
    torch.manual_seed(0)
    if net == "full":
        return MuZeroNetFull(785 * 4, 20).randomize_heads().to(dev).eval(), 20
    return MuZeroNet(193 * 4, 11).randomize_heads().to(dev).eval(), 11


def inputs(n, a, count, pinned):
    """`count` distinct tickets of device-resident (or pinned-host) inputs; hidden states in the pool's fp16."""
    rng = np.random.default_rng(n)
    out = []
    for k in range(count):
        legal = torch.from_numpy((rng.random((n, a)) < 0.6).astype(np.int32))
        legal[:, k % a] = 1
        t = dict(noise=torch.from_numpy(rng.dirichlet([0.3] * a, n).astype(np.float32)), reward=torch.zeros(n),
                 logits=torch.from_numpy(rng.standard_normal((n, a)).astype(np.float32)), legal=legal,
                 hidden=(torch.from_numpy(rng.standard_normal((n, 512)).astype(np.float32)).clamp_min(0) * 0.7).half(),
                 visits=torch.empty(n, a, dtype=torch.int32), values=torch.empty(n))
        if not pinned:
            t = {k2: v.to(dev) for k2, v in t.items()}
            t["visits"] = t["values"] = None       # results are read with stats() on the device
        else:
            t = {k2: v.pin_memory() for k2, v in t.items()}
        out.append(t)
    return out


def run(label, net, model, a, n, wave, depth, pinned, rep, profile=None):
    pipe = SearchPipeline(MCTS(SearchConfig(num_simulations=S, amp_type="torch_amp")), model, n, a, depth=depth,
                          wave=wave)
    tickets = inputs(n, a, 2 * wave, pinned)
    submit = lambda t: pipe.submit(0.25, t["noise"], t["reward"], t["logits"], t["legal"], t["hidden"], t["visits"],
                                   t["values"])
    for k in range(3 * depth * wave):          # every slot: eager search, capture, replay
        submit(tickets[k % len(tickets)])
    pipe.drain()
    torch.cuda.synchronize()
    count = max(TREES // n // wave, 2 * depth) * wave
    pipe.host_seconds, pipe.submitted = 0.0, 0
    ctx = profile if profile is not None else None
    t0 = time.perf_counter()
    if ctx is not None:
        ctx.__enter__()
    for k in range(count):
        last = submit(tickets[k % len(tickets)])
    pipe.drain()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if ctx is not None:
        ctx.__exit__(None, None, None)
    visits, _ = pipe.stats(last)
    assert int(visits.sum()) == n * (S - 1), "search result"
    rec = dict(label=label, net=net, n=n, wave=wave, depth=depth, inputs="pinned" if pinned else "device", rep=rep,
               executor=pipe.executor, tickets=count, window_s=round(dt, 4),
               sims_per_s=count * n * (S - 1) / dt, host_us_per_ticket=1e6 * pipe.host_seconds / pipe.submitted,
               profiled=ctx is not None)
    print(json.dumps(rec), flush=True)
    if ctx is None:
        with open(os.path.join(OUT, "wave.jsonl"), "a") as f:
            f.write(json.dumps(rec) + "\n")
    del pipe
    torch.cuda.synchronize()
    return rec


def summary(recs):
    rows = {}
    for r in recs:
        rows.setdefault((r["net"], r["inputs"], r["n"], r["label"]), []).append(r)
    print("net    inputs  n     config            M sims/s (median, min-max)   host us/ticket (median)")
    for (net, inp, n, label), rs in sorted(rows.items()):
        v = [r["sims_per_s"] / 1e6 for r in rs]
        h = [r["host_us_per_ticket"] for r in rs]
        print(f"{net:6s} {inp:7s} {n:5d} {label:17s} {statistics.median(v):8.1f} ({min(v):.1f}-{max(v):.1f})"
              f"            {statistics.median(h):8.1f}", flush=True)


if __name__ == "__main__":
    try:
        print(json.dumps(dict(device=torch.cuda.get_device_name(0), torch=torch.__version__,
                              cuda_device_max_connections=os.environ["CUDA_DEVICE_MAX_CONNECTIONS"])), flush=True)
        full, a_full = make_model("full")
        recs = []
        for rep in range(REPS):
            for n in (512, 1024, 2048):
                recs.append(run("a wave=1 depth=20", "full", full, a_full, n, 1, 20, False, rep))
                recs.append(run(f"b wave={4096 // n} depth=8", "full", full, a_full, n, 4096 // n, 8, False, rep))
        for rep in range(2):
            recs.append(run("a wave=1 depth=20", "full", full, a_full, 512, 1, 20, True, rep))
            recs.append(run("b wave=8 depth=8", "full", full, a_full, 512, 8, 8, True, rep))
        small, a_small = make_model("small")
        for rep in range(2):
            recs.append(run("a wave=1 depth=20", "small", small, a_small, 512, 1, 20, False, rep))
            recs.append(run("b wave=8 depth=8", "small", small, a_small, 512, 8, 8, False, rep))
        summary(recs)
        from torch.profiler import ProfilerActivity, profile
        TREES = 4096 * 32                      # a short window: tracing slows the host
        for tag, label, wave, depth in (("a", "a wave=1 depth=20", 1, 20), ("b", "b wave=8 depth=8", 8, 8)):
            prof = profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA])
            run(label, "full", full, a_full, 512, wave, depth, False, 0, profile=prof)
            prof.export_chrome_trace(os.path.join(OUT, f"wave_{tag}512.pt.trace.json"))
            table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=30)
            with open(os.path.join(OUT, f"wave_{tag}512_kernels.txt"), "w") as f:
                f.write(table)
            print(label, "\n", prof.key_averages().table(sort_by="cuda_time_total", row_limit=12), flush=True)
    except Exception:
        traceback.print_exc()
        sys.exit(1)
