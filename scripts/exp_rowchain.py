"""Experiment: the row-block resident network executor (hz_rowchain) against the cuBLASLt library chain (seven
launches; five for Hanabi-Small).
  1. parity of state / value / reward / policy logits (vs the library chain and vs a float64 evaluation)
  2. per-phase stamps of CTA 0
  3. time per chain alone (CUDA graph, back to back) and with D chains on D streams (what searches in flight see)
Env: N (rows, default 4096), D (streams, default 7), NET (full | small: MuZeroNetFull or the Hanabi-Small MuZeroNet,
default full)."""
import ctypes, os, sys, traceback
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from hanabizero_b200 import _lib
from hanabizero_b200.model import MuZeroNet, MuZeroNetFull
from hanabizero_b200.plan import BoundChain

dev = torch.device("cuda")
N = int(os.environ.get("N", "4096")); D = int(os.environ.get("D", "7")); NET = os.environ.get("NET", "full")
if NET not in ("full", "small"):
    sys.exit("NET must be full or small")
lib = _lib.load()
torch.manual_seed(0)
model = (MuZeroNetFull(785 * 4, 20) if NET == "full" else MuZeroNet(193 * 4, 11)).randomize_heads().to(dev).eval()
plan = model.recurrent_plan(torch.float16)
PHASES = 10 if NET == "full" else 6      # the job table's phases (hz_rowchain.cu)


def fill(ch, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    n = ch.n
    ch.x0.zero_()
    ch.x0[:, :plan.F].copy_((torch.randn(n, plan.F, device=dev, generator=g).clamp_min(0) * 0.7).half())
    a = torch.randint(0, plan.A, (n, 1), device=dev, generator=g)
    ch.x0[:, plan.F:].scatter_(1, a, 1.0)
    return a


def ref64(ch):
    w = {k: v.double() for k, v in plan._w.items()}
    x = ch.x0.double()
    relu = torch.relu
    H = plan.H
    if NET == "small":   # skip after bn1, no residual after fc3, one layer per head ([value | reward | policy])
        y1 = relu(x @ w["W1"].T + w["b1"] + x[:, :plan.F]); y2 = relu(y1 @ w["W2"].T + w["b2"]); s = relu(y2 @ w["W3"].T + w["b3"])
        h1 = relu(s @ w["Wh1"].T + w["bh1"])
        return s, torch.stack([h1[:, i * H:(i + 1) * H] @ w["WB3"][i].T + w["bB3"][i] for i in range(3)])
    y1 = relu(x @ w["W1"].T + w["b1"]); y2 = relu(y1 @ w["W2"].T + w["b2"]); s = relu(y2 @ w["W3"].T + w["b3"] + x[:, :plan.F])
    h1 = relu(s @ w["Wh1"].T + w["bh1"])
    a1 = relu(h1[:, :H] @ w["WB2"][0].T + w["bB2"][0]); v2 = relu(h1[:, H:2 * H] @ w["WB2"][1].T + w["bB2"][1])
    r2 = relu(h1[:, 2 * H:] @ w["WB2"][2].T + w["bB2"][2]); a2 = relu(a1 @ w["Wa2"].T + w["ba2"] + h1[:, :H])
    outs = [t @ w["WB3"][i].T + w["bB3"][i] for i, t in enumerate((v2, r2, a2))]
    return s, torch.stack(outs)


def parity(n):
    ch = BoundChain(plan, n)
    fill(ch, 1 + n)
    st = torch.cuda.current_stream().cuda_stream
    ch.bind_state(ch.state)
    ch.run(st); torch.cuda.synchronize()
    s_lib, o_lib = ch.state.clone(), ch.out.clone()
    s64, o64 = ref64(ch)
    ch.state.zero_(); ch.out.zero_()
    ch.set_executor("rows")
    print(f"n={n}: rows executor grid = {lib.hz_rowchain_grid(ch._rows)} CTAs", flush=True)
    ch.run(st); torch.cuda.synchronize()
    s_row, o_row = ch.state.clone(), ch.out.clone()
    ok = True
    for name, a, b, r in (("state", s_row, s_lib, s64), ("value logits", o_row[0], o_lib[0], o64[0]),
                          ("reward logits", o_row[1], o_lib[1], o64[1]), ("policy logits", o_row[2], o_lib[2], o64[2])):
        d = (a.double() - b.double()).abs(); e_row = (a.double() - r).abs().max().item(); e_lib = (b.double() - r).abs().max().item()
        scale = r.abs().max().item()
        bad = (d > 0.02 * max(scale, 1e-3)).sum().item()
        ok &= bad == 0 and e_row <= max(4 * e_lib, 0.01 * scale)
        print(f"  {name:14s} max|rows-lib| {d.max().item():.3e}  max|rows-f64| {e_row:.3e}  max|lib-f64| {e_lib:.3e}  "
              f"scale {scale:.3f}  elements off by > 2% of scale: {bad}", flush=True)
        if bad:
            idx = torch.nonzero(d > 0.02 * max(scale, 1e-3))[:6].tolist()
            print("     first offenders (row, col):", idx, flush=True)
    print(f"  parity n={n}: {'OK' if ok else 'FAILED'}", flush=True)
    return ch, ok


def stamps(ch):
    check = _lib.check
    check(lib.hz_rowchain_set_trace(ch._rows, 1))
    st = torch.cuda.current_stream().cuda_stream
    ch.run(st); torch.cuda.synchronize()
    g = lib.hz_rowchain_grid(ch._rows)
    buf = (ctypes.c_uint64 * (g * 40))()
    check(lib.hz_rowchain_read_trace(ch._rows, buf, g * 40))
    t = np.frombuffer(buf, dtype=np.uint64).reshape(g, 10, 4).astype(np.int64)
    check(lib.hz_rowchain_set_trace(ch._rows, 0))
    t0, last = t[0, 0, 0], PHASES - 1
    print("  CTA 0 stamps, ns from the first phase's start: [MMA may start, MMAs issued, accumulators complete, tile written]")
    for ph in range(PHASES):
        print(f"    phase {ph}: {(t[0, ph] - t0).tolist()}")
    print(f"  whole chain, CTA 0: {(t[0, last, 3] - t0) / 1e3:.1f} us; over CTAs: min {((t[:, last, 3] - t[:, 0, 0]).min()) / 1e3:.1f} "
          f"max {((t[:, last, 3] - t[:, 0, 0]).max()) / 1e3:.1f} us", flush=True)


def graph_of(ch, reps, stream):
    with torch.cuda.stream(stream):
        ch.run(stream.cuda_stream)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        for _ in range(reps):
            ch.run(torch.cuda.current_stream().cuda_stream)
    return g


def time_alone(ch, reps=49):
    s = torch.cuda.Stream()
    g = graph_of(ch, reps, s)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(s):
        g.replay(); g.replay()
        e0.record(s); g.replay(); g.replay(); e1.record(s)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (2 * reps)


def time_streams(chains, reps=49):
    streams = [torch.cuda.Stream() for _ in chains]
    graphs = [graph_of(c, reps, s) for c, s in zip(chains, streams)]
    e0 = torch.cuda.Event(enable_timing=True); ends = [torch.cuda.Event(enable_timing=True) for _ in chains]
    for s, g in zip(streams, graphs):
        with torch.cuda.stream(s):
            g.replay()
    torch.cuda.synchronize()
    e0.record()
    for s, g, e in zip(streams, graphs, ends):
        s.wait_event(e0)
        with torch.cuda.stream(s):
            g.replay(); g.replay(); e.record(s)
    torch.cuda.synchronize()
    return max(e0.elapsed_time(e) for e in ends) * 1e3 / (2 * reps * len(chains))


if __name__ == "__main__":
    try:
        _, ok_small = parity(128)
        _, ok_ragged = parity(300)
        ch, ok = parity(N)
        stamps(ch)
        if not (ok and ok_small and ok_ragged):
            print("PARITY FAILED - timings below are of a wrong kernel", flush=True)
        for n in sorted({512, 1024, N}):
            c = BoundChain(plan, n); fill(c, 7)
            t_lib = time_alone(c)
            c.set_executor("rows")
            t_row = time_alone(c)
            print(f"alone, n={n}: library {t_lib:.1f} us per chain, rows {t_row:.1f} us per chain", flush=True)
        for n, d in ((N, D), (512, 8), (512, 16), (1024, 8)):
            chains = [BoundChain(plan, n) for _ in range(d)]
            for c in chains:
                fill(c, 3)
            t_lib = time_streams(chains)
            for c in chains:
                c.set_executor("rows")
            t_row = time_streams(chains)
            print(f"{d} streams, n={n}: library {t_lib:.2f} us per chain (aggregate), rows {t_row:.2f} us per chain", flush=True)
    except Exception:
        traceback.print_exc()
        sys.exit(1)
