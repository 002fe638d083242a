#!/usr/bin/env python
"""Benchmark of the HanabiZero self-play hot path (BASELINE.json metric: MCTS simulations/s and
Hanabi env steps/s on 1/2/4/8 B200 next to the reference's host-CPU implementation).

    python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path on the host cores
    python bench.py --config {1..5}                          # BASELINE.json configs[0..4]; default 4
    python bench.py --scaling weak                           # `trees_total` of the config PER GPU instead of in total
    python bench.py --dump-outputs DIR                       # + root visits / values of the last timed search as DIR/*.npy

A "step" is one batched search: Roots.prepare + MCTS.run_multi (num_simulations-1 simulations, the
PyTorch network included, random-init weights with re-drawn heads) + root statistics.  The default is
BASELINE.json configs[3] AS WRITTEN: 4096 Hanabi-Full trees x 50 simulations IN TOTAL, the root batch sharded
over the N GPUs (strong scaling: 4096 / N trees per GPU, one model replica per GPU, one NCCL all_gather of the
final statistics per search, issued off the compute stream).  With N > 1 the line also carries a `weak` object
(the same search with 4096 trees PER GPU).  `value` = simulations/s of the whole job with inputs resident in
HBM; `e2e` = the same through the public host-facing API with pinned host inputs copied in and statistics copied
out inside the timed region.  The Hanabi env is timed the same way and reported in the `env` object.  One JSON
line is printed by rank 0.
"""
import argparse
import json
import multiprocessing as mp
import os
# more than 8 searches in flight need more than the default 8 hardware work queues, or streams that share a queue
# serialise (small root batches: 512 trees x 20 searches 47 -> 81 M simulations/s); must be set before CUDA starts
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CONST = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.999, delta=0.006, frac=0.25)
F_HIDDEN = 512

# BASELINE.json configs[0..4] (SURVEY.md §8d)
CONFIGS = {
    1: dict(game="Hanabi-Small", mdp="global", trees_total=16, sims=50,
            name="config 1: Hanabi-Small 2p global MDP, p_mcts_num=16 trees x 50 simulations"),
    2: dict(game="Hanabi-Full", mdp="global", trees_total=256, sims=50,
            name="config 2: Hanabi-Full 2p global MDP, 256 trees x 50 simulations"),
    3: dict(game="Hanabi-Full", mdp="local", trees_total=1024, sims=50,
            name="config 3: Hanabi-Full 2p local POMDP, stack=4, 1024 trees x 50 simulations"),
    4: dict(game="Hanabi-Full", mdp="global", trees_total=4096, sims=50,
            name="config 4: Hanabi-Full 2p global MDP, 4096 trees x 50 simulations"),
    5: dict(game="Hanabi-Full", mdp="global", trees_total=16384, sims=200,
            name="config 5: Hanabi-Full 2p global MDP, 16384 trees x 200 simulations (deep-tree stress)"),
}
GAMES = {"Hanabi-Full": dict(actions=20, glob=785, loc=660), "Hanabi-Small": dict(actions=11, glob=193, loc=173)}


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--config", type=int, default=4, choices=sorted(CONFIGS), help="BASELINE.json configs[n-1]")
    p.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                   help="strong: the config's trees in TOTAL, sharded over the GPUs; weak: that many PER GPU")
    p.add_argument("--trees-total", type=int, default=None, help="override the config's total tree count")
    p.add_argument("--trees", type=int, default=None, help="trees (and games) PER GPU (implies --scaling weak)")
    p.add_argument("--sims", type=int, default=None)
    p.add_argument("--stack", type=int, default=4)
    p.add_argument("--amp", default="torch_amp", choices=["torch_amp", "none"])
    p.add_argument("--mdp", default=None, choices=["global", "local"], help="observation fed to the network")
    p.add_argument("--env-steps", type=int, default=200, help="env steps per timed env pass")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-graph", action="store_true")
    p.add_argument("--sm-target", type=int, default=None,
                   help="SMs each in-flight search's library GEMMs are sized for (default: SearchPipeline's rule; 0 = whole device)")
    p.add_argument("--stage-limit", type=int, default=None,
                   help="hz_search_io.stage_limit of the in-flight searches (default: SearchPipeline's, 4; 0 = stage all that fits)")
    p.add_argument("--executor", default="auto", choices=["auto", "library", "rows"],
                   help="network executor of the in-flight searches: seven cuBLASLt launches or the row-block resident "
                        "kernel (auto = SearchPipeline's choice: rows when searches overlap)")
    p.add_argument("--in-flight", type=int, default=None,
                   help="independent searches kept in flight per GPU (SearchPipeline depth); 1 = one search at a time")
    p.add_argument("--quick", action="store_true", help="search + roofline only (skip env / self-play / extras)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the root statistics of the last timed search (the `value` path) as DIR/<name>.npy")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        p.error("--dump-outputs writes what the GPU path computes: it needs --impl ours")
    return args


def resolve_workload(args, world):
    """-> dict(game, A, mdp, sims, scaling, per_gpu, total, name): what one step of this run searches."""
    c = dict(CONFIGS[args.config])
    if args.sims is not None:
        c["sims"] = args.sims
    if args.mdp is not None:
        c["mdp"] = args.mdp
    scaling = args.scaling
    if args.trees is not None:
        scaling, per = "weak", args.trees
    elif scaling == "weak":
        per = args.trees_total or c["trees_total"]
    else:
        total = args.trees_total or c["trees_total"]
        if total % world:
            raise SystemExit(f"{total} trees do not shard evenly over {world} GPUs")
        per = total // world
    g = GAMES[c["game"]]
    return dict(game=c["game"], A=g["actions"], mdp=c["mdp"], obs_dim=g["glob"] if c["mdp"] == "global" else g["loc"],
                sims=c["sims"], scaling=scaling, per_gpu=per, total=per * world, name=c["name"], config=args.config)


def b_sim(A, D, s, F):
    """Algorithmic bytes of one simulation of one tree (SURVEY.md §8d); F = hidden row in 4-byte units."""
    return D * (16 * A + 32) + 22 * A + 20 * (D + 1) + 12 * s + 32 + 8 * F


def b_env_step(obs_dim, A, obs_bytes):
    """Algorithmic bytes of one env step of one game (SURVEY.md §8d): state r/w + the observation in the dtype
    that is actually written + legal mask + reward/done/score."""
    return 2 * 192 + obs_bytes * obs_dim + obs_bytes * A + 12


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Writes each array (same row count, float32/float64) as path/<name>.npy, so that two builds run with the same
    arguments can be compared output for output.  Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of the rows is
    written (the same rows in every run) and `rows.npy` holds their indices."""
    os.makedirs(path, exist_ok=True)
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a.nbytes for a in arrays.values()) // max(n, 1)
    if n * row_bytes > DUMP_LIMIT_BYTES:
        keep = (DUMP_LIMIT_BYTES - 4096) // (row_bytes + 8)        # + the float64 row index; 4 KB for the .npy headers
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = dict({k: a[rows] for k, a in arrays.items()}, rows=rows.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ======================================================================================================
# CPU reference arm (test infrastructure: the ONLY place besides tests/smoke that executes oracle/)
# ======================================================================================================
def _load_ref_cytree():
    import importlib.util
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    so = [f for f in os.listdir(ref_dir) if f.startswith("cytree.") and f.endswith(".so")] if os.path.isdir(ref_dir) else []
    if not so:
        return None
    spec = importlib.util.spec_from_file_location("cytree", os.path.join(ref_dir, so[0]))
    tree = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tree)
    return tree


def _ref_tree_worker(args):
    """One reference actor: the loop of core/mcts.py:24-55 around the reference's own cytree module
    (oracle/_ref, stock build) with pre-generated network outputs instead of the GPU model —
    Python-list marshalling, host hidden-state gather and .tolist() included, as the reference pays."""
    n, A, S, seed, reps = args
    tree = _load_ref_cytree()
    kind = "reference" if tree is not None else "port"
    rng = np.random.default_rng(seed)
    logits0 = rng.standard_normal((n, A)).astype(np.float32)
    noise = rng.dirichlet([0.3] * A, n).astype(np.float32)
    mask = np.ones((n, A), np.float64)
    hidden_roots = rng.standard_normal((n, F_HIDDEN)).astype(np.float32)
    sim_hidden = rng.standard_normal((n, F_HIDDEN)).astype(np.float32)
    sim_out = [(rng.standard_normal((n, 1)).astype(np.float32), rng.standard_normal((n, 1)).astype(np.float32),
                rng.standard_normal((n, A)).astype(np.float32)) for _ in range(4)]
    t0 = time.perf_counter()
    for _ in range(reps):
        if tree is not None:
            roots = tree.Roots(n, A, S)
            roots.prepare(CONST["frac"], noise.tolist(), [0.0] * n, logits0.tolist(), [m for m in mask])
            pool = [hidden_roots]
            mm = tree.MinMaxStatsList(n)
            mm.set_delta(CONST["delta"])
            for x in range(1, S):
                results = tree.ResultsWrapper(n)
                ix, iy, la = tree.multi_traverse(roots, CONST["pb_c_base"], CONST["pb_c_init"], CONST["discount"], mm, results)
                hs = np.asarray([pool[a][b] for a, b in zip(ix, iy)])       # core/mcts.py:31-33
                la = np.asarray(la)
                value, reward, pol = sim_out[x % 4]
                reward_pool = reward.reshape(-1).tolist()
                value_pool = value.reshape(-1).tolist()
                pol = pol.copy()
                pol[np.isnan(pol)] = 0.0
                pool.append(sim_hidden)
                tree.multi_back_propagate(x, CONST["discount"], reward_pool, value_pool, pol.tolist(), mm, results)
            roots.get_distributions(); roots.get_values()
        else:
            from oracle import loader as L
            eng = L.oracle_tree(n, A, S, CONST["delta"])
            eng.prepare(CONST["frac"], noise, np.zeros(n, np.float32), logits0, mask.astype(np.int32))
            for x in range(1, S):
                eng.traverse(CONST["pb_c_base"], CONST["pb_c_init"], CONST["discount"])
                value, reward, pol = sim_out[x % 4]
                eng.backprop(x, CONST["discount"], reward.reshape(-1), value.reshape(-1), pol)
            eng.stats()
    return time.perf_counter() - t0, kind


def _ref_env_worker(args):
    """The reference's libhanabi in a C++ loop (apply + deal + 2x observe/encode per step, random legal play)."""
    n_steps, seed, preset = args
    from oracle import loader as L
    kind = "reference" if L.have_ref() else "port"
    g = L.ref_hanabi(preset, seed) if kind == "reference" else L.oracle_hanabi(preset, seed)
    t0 = time.perf_counter()
    g.play(n_steps, seed + 1)
    return time.perf_counter() - t0, kind


def _ref_pyenv_worker(args):
    """The reference's Python API (envs/hanabi/rl_env.py:148-442 HanabiEnv.reset/step over pyhanabi.py + cffi +
    libpyhanabi.so, byte-compiled unmodified into oracle/_ref/refpy): what the reference's callers actually pay
    per env step.  Random legal play, episodes reset as they end."""
    n_steps, seed, game = args
    from oracle import refpy
    if not refpy.available():
        return None
    env = refpy.load_env_class()({"hanabi_name": game, "seed": seed})
    rng = np.random.default_rng(seed)
    legal = np.asarray(env.reset()[2])
    t0 = time.perf_counter()
    for _ in range(n_steps):
        out = env.step(int(rng.choice(np.flatnonzero(legal))))
        legal = np.asarray(out[5])
        if out[3]:
            legal = np.asarray(env.reset()[2])
    return time.perf_counter() - t0


def cpu_reference(trees, A, S, cores, reps=1, env_steps_per_core=20000, game="Hanabi-Full", pyenv_steps_per_core=0):
    """Reference CPU path on `cores` processes (mirrors num_actors: the reference's only parallelism)."""
    ctx = mp.get_context("spawn")
    n_proc = max(1, min(cores, trees))
    per = [trees // n_proc + (1 if i < trees % n_proc else 0) for i in range(n_proc)]
    preset = 0 if game == "Hanabi-Full" else 1
    with ctx.Pool(cores) as pool:
        res = pool.map(_ref_tree_worker, [(p, A, S, 100 + i, reps) for i, p in enumerate(per)])
        wall = max(max(r[0] for r in res), 1e-9)
        sims_s = trees * (S - 1) * reps / wall
        eres = pool.map(_ref_env_worker, [(env_steps_per_core, i, preset) for i in range(cores)])
        env_s = env_steps_per_core * cores / max(r[0] for r in eres)
        py_s = None
        if pyenv_steps_per_core:
            pres = pool.map(_ref_pyenv_worker, [(pyenv_steps_per_core, i, game) for i in range(cores)])
            if all(r is not None for r in pres):
                py_s = pyenv_steps_per_core * cores / max(pres)
    return dict(sims_per_s=sims_s, env_steps_per_s=env_s, pyenv_steps_per_s=py_s, kind=res[0][1], env_kind=eres[0][1],
                cores=cores, tree_procs=n_proc, wall_s=wall)


def reference_with_model(trees, A, S, game="Hanabi-Full", obs_dim=785):
    """Informational: the loop of core/mcts.py:24-55 exactly as the reference runs it — its own cytree on the
    host, the PyTorch network on the GPU, Python-list marshalling, host hidden-state gather, H2D of the batch
    and D2H of the outputs EVERY simulation (one actor process).  Returns simulations/s or None."""
    try:
        import torch
        if not torch.cuda.is_available():
            return None
        tree = _load_ref_cytree()
        if tree is None:
            return None
        from hanabizero_b200.model import MuZeroNet, MuZeroNetFull
        torch.manual_seed(0)
        net = MuZeroNetFull if game == "Hanabi-Full" else MuZeroNet
        model = net(obs_dim * 4, A).randomize_heads(seed=0).cuda().eval()
        rng = np.random.default_rng(0)
        obs = torch.from_numpy((rng.random((trees, obs_dim * 4)) < 0.2).astype(np.float32)).cuda()
        best = None
        for rep in range(2):
            with torch.no_grad():
                with torch.autocast("cuda", dtype=torch.float16):
                    out = model.initial_inference(obs)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                roots = tree.Roots(trees, A, S)
                noises = [rng.dirichlet([0.3] * A).astype(np.float32).tolist() for _ in range(trees)]
                roots.prepare(CONST["frac"], noises, out.reward, out.policy_logits.tolist(), [np.ones(A) for _ in range(trees)])
                pool = [out.hidden_state]
                mm = tree.MinMaxStatsList(trees)
                mm.set_delta(CONST["delta"])
                for x in range(1, S):
                    results = tree.ResultsWrapper(trees)
                    ix, iy, la = tree.multi_traverse(roots, CONST["pb_c_base"], CONST["pb_c_init"], CONST["discount"], mm, results)
                    hs = torch.from_numpy(np.asarray([pool[a][b] for a, b in zip(ix, iy)])).to("cuda")
                    la = torch.from_numpy(np.asarray(la)).to("cuda").unsqueeze(1).long()
                    with torch.autocast("cuda", dtype=torch.float16):
                        no = model.recurrent_inference(hs.float(), la)
                    pol = no.policy_logits
                    pol[np.isnan(pol)] = 0.0
                    pool.append(no.hidden_state)
                    tree.multi_back_propagate(x, CONST["discount"], no.reward.reshape(-1).tolist(),
                                              no.value.reshape(-1).tolist(), pol.tolist(), mm, results)
                roots.get_distributions(); roots.get_values()
                dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        return trees * (S - 1) / best
    except Exception as e:  # informational only
        return f"unavailable: {type(e).__name__}: {e}"


def config_obj(args, wl, world):
    """The `config` object both arms print (same workload, same words): what is searched, not how."""
    S, per = wl["sims"], wl["per_gpu"]
    nodes_mb = per * (S + 1) * wl["A"] * 16 / 1e6
    pool_mb = per * S * F_HIDDEN * (2 if args.amp == "torch_amp" else 4) / 1e6
    return {"workload": f"{wl['name']}: {wl['total']} trees in total, {per} per GPU x {world} GPU(s) ({wl['scaling']} scaling), "
                        f"{S - 1} simulations executed per search (core/mcts.py:25-26)",
            "baseline_config": wl["config"], "trees_per_gpu": per, "trees_total": wl["total"], "actions": wl["A"],
            "simulations": S, "stack": args.stack, "mdp": wl["mdp"],
            "l2": f"per search the tree nodes ({nodes_mb:.0f} MB) + hidden pool ({pool_mb:.0f} MB) per GPU "
                  f"{'exceed' if nodes_mb + pool_mb > 126 else 'fit'} the 126 MB L2; the GPU arm's roofline launches are timed "
                  "with L2 flushed (256 MiB write) before each one"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    wl = resolve_workload(args, max(args.gpus, 1))
    A, S, trees = wl["A"], wl["sims"], wl["total"]
    # a step = one search of the whole job's root batch on the host cores; small batches are repeated so that a
    # step lasts long enough to time (the repeat count is part of the sample description)
    reps = max(1, int(round(2e5 / max(trees * (S - 1), 1))))
    times = []
    out = None
    for i in range(args.warmup + args.steps):
        out = cpu_reference(trees, A, S, cores, reps=reps, env_steps_per_core=5000, game=wl["game"],
                            pyenv_steps_per_core=300 if i == args.warmup + args.steps - 1 else 0)
        if i >= args.warmup:
            times.append(out)
    val = statistics.mean(t["sims_per_s"] for t in times)
    env = statistics.mean(t["env_steps_per_s"] for t in times)
    sample = (f"{trees} {wl['game']} trees x {S - 1} simulations (x{reps} repeats) per step split over {out['tree_procs']} "
              "processes; reference cytree driven like core/mcts.py with pre-generated network outputs (no model time); "
              f"env: {5000 * out['cores']} steps of reference libhanabi (apply+deal+2x observe/encode), random legal play; "
              f"env_python_api: {300 * out['cores']} steps of the reference's HanabiEnv.step (rl_env.py) over {out['cores']} processes")
    line = {
        "impl": "reference", "metric": "mcts_simulations_per_sec", "value": val, "unit": "simulations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * trees * (S - 1) / val, "higher_is_better": True, "scaling": wl["scaling"],
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_obj(args, wl, max(args.gpus, 1)),
        "cpu_baseline": {"value": val, "unit": "simulations/s", "cores": out["cores"], "kind": out["kind"], "sample": sample},
        "e2e": {"value": val, "unit": "simulations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "env": {"metric": "hanabi_env_steps_per_sec", "value": env, "unit": "steps/s", "kind": out["env_kind"],
                "cores": out["cores"], "python_api_steps_per_s": out["pyenv_steps_per_s"]},
        "gpu_launches": 0,
        "reference_with_model_on_gpu": {
            "value": reference_with_model(min(trees, 1024), A, S, wl["game"], wl["obs_dim"]), "unit": "simulations/s",
            "what": "informational: one reference actor, its own cytree on the host + the PyTorch network on cuda:0 with "
                    "per-simulation H2D/D2H and list marshalling exactly as core/mcts.py:24-55 does, "
                    f"{min(trees, 1024)} trees x {S - 1} simulations"},
    }
    print(json.dumps(line), flush=True)


# ======================================================================================================
# our arm
# ======================================================================================================
class ClockSampler(threading.Thread):
    """One long-running `nvidia-smi -lms 100` for the whole timed phase (the recipe's clocks line)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                parts = [x.strip() for x in line.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        self.join(timeout=3)
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": float(self.samples[0][1]) if self.samples else None,
                "samples": len(self.samples), "reasons": sorted(reasons)}


def ncu_env_traffic_per_launch(games):
    """The same for the env kernel (profiles/r<NN>_ncu_full_k_env_<games>.csv, caches left warm)."""
    import csv
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", f"r*_ncu_full_k_env_{games}.csv")), reverse=True):
        try:
            rows = list(csv.reader(open(path)))
            hdr, units = rows[0], rows[1]
            ir, iw, ik = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum"), hdr.index("Kernel Name")
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            vals = [float(r[ir]) * scale[units[ir]] + float(r[iw]) * scale[units[iw]] for r in rows[2:] if "k_env" in r[ik]]
            if vals:
                return sum(vals) / len(vals), os.path.basename(path)
        except Exception:
            continue
    return None, None


def ncu_traffic_per_launch(trees, stage_limit=0):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the fused search-step kernel, from the newest
    committed `ncu --set full` capture of that kernel at this tree count under profiles/
    (r<NN>_ncu_full_k_search_step_<trees>.csv; captured with the caches left warm, as inside a search: the same capture
    with ncu's default cache flush is the *_cold.csv next to it); (None, None) if there is none."""
    import csv
    import glob
    suffix = f"_stage_limit{stage_limit}" if stage_limit else ""
    paths = [p for p in glob.glob(os.path.join(ROOT, "profiles", f"r*_ncu_full_k_search_step_{trees}{suffix}.csv"))]
    for path in sorted(paths, reverse=True):
        try:
            rows = list(csv.reader(open(path)))
            hdr, units = rows[0], rows[1]
            ir, iw, ik = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum"), hdr.index("Kernel Name")
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            vals = [float(r[ir]) * scale[units[ir]] + float(r[iw]) * scale[units[iw]] for r in rows[2:]
                    if "k_search_step" in r[ik]]
            if vals:
                return sum(vals) / len(vals), os.path.basename(path)
        except Exception:
            continue
    return None, None


class SearchBench:
    """Everything one rank needs to time searches of `n` trees: roots from real Hanabi positions, the model, the
    device-resident step and the host-facing (end-to-end) steps."""

    def __init__(self, torch, args, wl, n, rank, world, dev, model):
        from hanabizero_b200 import cytree
        from hanabizero_b200.dist import AsyncStatsGather
        from hanabizero_b200.hanabi_env import HanabiVecEnv
        from hanabizero_b200.mcts import MCTS, SearchConfig
        self.torch, self.cytree, self.args, self.wl = torch, cytree, args, wl
        self.n, self.rank, self.world, self.dev, self.model = n, rank, world, dev, model
        A, S = wl["A"], wl["sims"]
        self.A, self.S = A, S
        self.cfg = SearchConfig(num_simulations=S, amp_type=args.amp)
        # synthetic roots: real Hanabi positions (reset + 10 random legal steps) -> initial inference
        self.env = HanabiVecEnv(n, wl["game"], np.arange(n) + rank * n, device=dev)
        g, loc, legal = self.env.reset_all()
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        for _ in range(10):
            acts = torch.multinomial(legal, 1, generator=gen).view(-1).int()
            g, loc, legal, _, _, _ = self.env.step_all(acts, auto_reset=True)
        self.env.check()
        obs = (g if wl["mdp"] == "global" else loc).repeat(1, args.stack)
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=args.amp == "torch_amp"):
            _, root_logits, root_hidden = model.initial_inference_device(obs)
        self.root_logits = root_logits.float().contiguous()
        self.root_hidden = root_hidden.contiguous()
        rng = np.random.default_rng(7 + rank)
        self.noise = torch.from_numpy(rng.dirichlet([0.3] * A, n).astype(np.float32)).to(dev)
        self.zeros_r = torch.zeros(n, device=dev)
        self.legal = legal
        self.legal_i = legal.int().contiguous()
        self.gather = AsyncStatsGather(n, A, dev, depth=2) if world > 1 else None
        self.mcts = MCTS(self.cfg)
        self.holder = [None]
        self.ticket = None
        self.pipe, self.pipe_ticket = None, None

    def pipelined_step(self):
        """The same search through SearchPipeline with device-resident inputs: `--in-flight` independent searches on
        their own streams (and the statistics all_gather of each, off the compute streams)."""
        if self.pipe is None:
            from hanabizero_b200.dist import AsyncStatsGather
            from hanabizero_b200.mcts import SearchPipeline
            depth = max(1, self.args.in_flight)
            gather = AsyncStatsGather(self.n, self.A, self.dev, depth=depth) if self.world > 1 else None
            self.pipe = SearchPipeline(self.mcts, self.model, self.n, self.A, depth=depth, device=self.dev, gather=gather,
                                       gemm_sm_target=self.args.sm_target, stage_limit=self.args.stage_limit,
                                       executor=self.args.executor)
        self.pipe_ticket = self.pipe.submit(CONST["frac"], self.noise, self.zeros_r, self.root_logits, self.legal_i,
                                            self.root_hidden)
        return self.pipe_ticket

    def finish_pipeline(self):
        """Drain the pipeline; returns (visits, values) of the last search and all ranks' statistics of it (or None)."""
        self.pipe.drain()
        stats = self.pipe.stats(self.pipe_ticket)
        return stats, (self.pipe.gathered(self.pipe_ticket) if self.pipe.gather is not None else None)

    def search_step(self, executor=None, use_graph=None):
        """Roots.prepare + run_multi + root statistics (+ the statistics all_gather, off the compute stream).  One search
        at a time runs the library chain (its lower latency) unless --executor rows asks otherwise."""
        if executor is None:
            executor = "rows" if self.args.executor == "rows" else "library"
        roots = self.cytree.Roots(self.n, self.A, self.S, device=self.dev)
        roots.prepare(CONST["frac"], self.noise, self.zeros_r, self.root_logits, self.legal_i)
        self.mcts.run_multi(roots, self.model, self.root_hidden, executor=executor,
                            use_graph=(not self.args.no_graph) if use_graph is None else use_graph)
        visits, values = roots.get_stats_tensors()
        if self.gather is not None:
            self.ticket = self.gather.submit(visits, values)
        self.holder[0] = roots
        return visits, values

    def finish(self):
        """All ranks' statistics of the last search (waits for the in-flight gather on the current stream)."""
        if self.gather is not None and self.ticket is not None:
            return self.gather.result(self.ticket)
        return None


def run_ours(args):
    import torch
    import torch.distributed as dist
    from hanabizero_b200 import _lib, cytree
    from hanabizero_b200.hanabi_env import HanabiVecEnv
    from hanabizero_b200.mcts import MCTS, SearchPipeline
    from hanabizero_b200.model import MuZeroNet, MuZeroNetFull

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: hanabizero_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    wl = resolve_workload(args, world)
    N, A, S, F = wl["per_gpu"], wl["A"], wl["sims"], F_HIDDEN
    K, W = args.steps, max(args.warmup, 3)
    # searches in flight: at most --in-flight, lowered so that the K timed searches split into equally full waves (a ragged
    # last wave would run with fewer searches in flight than the figure claims)
    if args.in_flight is None:
        # a search is a chain of ~60-70 us steps whatever its size: small root batches (the shards of a strongly scaled
        # job) need more searches in flight to fill the GPU than 4096-tree ones
        rows_ok = wl["game"] == "Hanabi-Full" and args.amp == "torch_amp" and args.executor != "library"
        args.in_flight = 20 if (N < 3072 and rows_ok) else 8
    if args.in_flight > 1:
        waves = -(-K // args.in_flight)
        args.in_flight = max(1, -(-K // waves))
    torch.manual_seed(0)
    net = MuZeroNetFull if wl["game"] == "Hanabi-Full" else MuZeroNet
    model = net(wl["obs_dim"] * args.stack, A).randomize_heads(seed=0).to(dev).eval()
    sb = SearchBench(torch, args, wl, N, rank, world, dev, model)
    env, cfg, mcts = sb.env, sb.cfg, sb.mcts

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def time_searches(bench, steps, warm, piped=False):
        """CUDA-event time of `steps` searches of one SearchBench (barrier + synchronize on both sides, max over
        ranks); the gather of the last search is inside the timed region.  piped: through SearchPipeline with
        `--in-flight` searches on their own streams (drained inside the timed region), else one search at a time.
        -> (ms, (visits, values) of the last search, all ranks' statistics of it or None)."""
        if piped:
            for _ in range(max(warm, 3 * args.in_flight)):    # each slot: one eager search, one capture, one replay
                bench.pipelined_step()
            bench.finish_pipeline()
            bench.pipe.host_seconds, bench.pipe.submitted = 0.0, 0     # host time per submit: timed searches only
            barrier()
            e0.record()
            for _ in range(steps):
                bench.pipelined_step()
            stats, out = bench.finish_pipeline()              # host-blocking: every slot's search and gather is done
            e1.record()
            barrier()
            return max_over_ranks(e0.elapsed_time(e1)), stats, out
        for _ in range(warm):
            bench.search_step()
        bench.finish()
        barrier()
        e0.record()
        for _ in range(steps):
            stats = bench.search_step()
        out = bench.finish()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)), stats, out

    launches_before, gemm_before = _lib.launch_count(), _lib.gemm_launch_count()
    sb.search_step()                       # eager search (also the launch census)
    torch.cuda.synchronize()
    launches_per_search = _lib.launch_count() - launches_before
    gemm_per_search = _lib.gemm_launch_count() - gemm_before
    launches_one, gemm_one = launches_per_search, gemm_per_search
    piped_executor = ("rows" if args.in_flight > 1 else "library") if args.executor == "auto" else args.executor
    if args.in_flight > 1 and piped_executor == "rows":
        # the timed searches run the network on the row-block resident executor: census of that path (eager, no graph)
        launches_before, gemm_before = _lib.launch_count(), _lib.gemm_launch_count()
        sb.search_step(executor="rows", use_graph=False)
        torch.cuda.synchronize()
        launches_per_search = _lib.launch_count() - launches_before
        gemm_per_search = _lib.gemm_launch_count() - gemm_before

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)   # let nvidia-smi attach before the timed regions
    # ---- timed region 1: device-resident search ------------------------------------------------
    piped = args.in_flight > 1
    ms_one, (visits_one, _), _ = time_searches(sb, K, W)             # one search at a time (the latency figure)
    sims_total = world * N * (S - 1) * K
    value_one = sims_total / (ms_one * 1e-3)
    if piped:
        ms_total, (visits, values), gathered = time_searches(sb, K, W, piped=True)
        # same inputs: identical trees when the pipeline runs the same library kernels; with GEMMs sized for a share of
        # the SMs the network roundings differ in the last bits, so only the simulation count is checked then
        assert sb.pipe.gemm_sm_target != 0 or sb.pipe.executor != "library" or torch.equal(visits, visits_one), "a search in the pipeline must equal the same search run alone"
        assert int(visits.sum().item()) == N * (S - 1)
    else:
        ms_total, (visits, values), gathered = time_searches(sb, K, W)
    value = sims_total / (ms_total * 1e-3)
    assert int(visits.sum().item()) == N * (S - 1), "search did not run the expected simulations"
    if gathered is not None:
        assert gathered[0].shape[0] == world * N and torch.equal(gathered[0][rank * N:(rank + 1) * N], visits), \
            "gathered root statistics do not contain this rank's shard"
    if args.dump_outputs and rank == 0:
        # now, before later phases reuse the pipeline's statistics buffers; every rank's shard when there are several
        out_visits, out_values = gathered if gathered is not None else (visits, values)
        dump_outputs(args.dump_outputs, {"root_visits": out_visits.cpu().numpy().astype(np.float32),
                                         "root_values": out_values.cpu().numpy().astype(np.float32)})

    # with more than one GPU: the same search with the config's tree count PER GPU (weak scaling), for the record
    weak = None
    if world > 1 and wl["scaling"] == "strong" and not args.quick:
        wl_w = dict(wl, per_gpu=wl["total"], total=wl["total"] * world, scaling="weak")
        sbw = SearchBench(torch, args, wl_w, wl_w["per_gpu"], rank, world, dev, model)
        kw = K if piped else max(K // 2, 3)      # whole waves of the pipeline
        ms_w, _, _ = time_searches(sbw, kw, 3, piped=piped)
        weak = {"value": wl_w["total"] * (S - 1) * kw / (ms_w * 1e-3), "unit": "simulations/s", "trees_per_gpu": wl_w["per_gpu"],
                "trees_total": wl_w["total"], "ms_per_step": ms_w / kw, "steps": kw}
        del sbw

    # ---- timed region 2: end to end through the host-facing API with pinned host buffers ----------------
    noise, root_logits, root_hidden, legal_i = sb.noise, sb.root_logits, sb.root_hidden, sb.legal_i
    h_noise, h_logits = noise.cpu().pin_memory(), root_logits.cpu().pin_memory()
    h_legal, h_hidden = legal_i.cpu().pin_memory(), root_hidden.cpu().pin_memory()
    h_reward = torch.zeros(N).pin_memory()
    h_visits = torch.empty(N, A, dtype=torch.int32).pin_memory()
    h_values = torch.empty(N).pin_memory()

    def e2e_step():
        roots = cytree.Roots(N, A, S, device=dev)
        roots.prepare(CONST["frac"], h_noise, h_reward, h_logits, h_legal)
        mcts.run_multi(roots, model, h_hidden, use_graph=not args.no_graph)
        v, val = roots.get_stats_tensors()
        h_visits.copy_(v, non_blocking=True)
        h_values.copy_(val, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        sb.holder[0] = roots
        return h_visits

    def timed_e2e(step_fn, finish=None, warm=2):
        for _ in range(warm):
            step_fn()
        if finish:
            finish()
        barrier()
        e0.record()
        for _ in range(K):
            step_fn()
        if finish:
            finish()
        e1.record()
        barrier()
        return sims_total / (max_over_ranks(max(e0.elapsed_time(e1), 0.0)) * 1e-3)

    e2e_serial = timed_e2e(e2e_step, warm=6)   # new Roots per search alternate between two cached handles: eager, capture, replay each
    # the same work through the double-buffered public API: the copies of neighbouring searches overlap the search
    depth = max(args.in_flight, 2)
    pipe = sb.pipe if (sb.pipe is not None and world == 1) else SearchPipeline(mcts, model, N, A, depth=depth, device=dev,
                                                                               gemm_sm_target=args.sm_target,
                                                                               stage_limit=args.stage_limit,
                                                                               executor=args.executor)
    depth = pipe.depth
    h_out = [(torch.empty(N, A, dtype=torch.int32).pin_memory(), torch.empty(N).pin_memory()) for _ in range(depth)]
    turn = [0]

    def piped_step():
        hv, hval = h_out[turn[0] % depth]
        turn[0] += 1
        pipe.submit(CONST["frac"], h_noise, h_reward, h_logits, h_legal, h_hidden, hv, hval)

    e2e_value = timed_e2e(piped_step, pipe.drain, warm=3 * depth)   # each slot: one eager search, one capture, one replay
    assert int(h_out[0][0].sum().item()) == N * (S - 1) and torch.equal(h_out[0][0], h_out[1][0]), "pipelined search result"
    assert pipe.gemm_sm_target != 0 or pipe.executor != "library" or torch.equal(h_out[0][0], h_visits), "pipelined and serial searches must agree"
    h2d = sum(t.numel() * t.element_size() for t in (h_noise, h_logits, h_legal, h_hidden, h_reward))
    d2h = h_visits.numel() * 4 + h_values.numel() * 4

    # ---- plan path vs nn.Module path: do the two ways of running the SAME network pick the same moves? -------
    agreement = None
    if rank == 0 and not args.quick and N * S <= 4096 * 50:
        roots_m = cytree.Roots(N, A, S, device=dev)
        roots_m.prepare(CONST["frac"], noise, sb.zeros_r, root_logits, legal_i)
        MCTS(cfg, use_plan=False).run_multi(roots_m, model, root_hidden, use_graph=False)
        vm, valm = roots_m.get_stats_tensors()
        vp = h_visits.to(dev)
        agreement = {"root_action_agreement": float((vm.argmax(1) == vp.argmax(1)).float().mean()),
                     "visit_count_l1_per_tree": float((vm - vp).abs().sum(1).float().mean()),
                     "root_value_max_abs_diff": float((valm - h_values.to(dev)).abs().max()),
                     "what": "arg-max root action of the production path (BN-folded fp16 GEMM plan + fused tree step) vs the "
                             "nn.Module path (PyTorch autocast kernels + generic tree calls) on the same roots and noise; the "
                             "trees are bit-exact functions of the network outputs, the difference is network rounding"}
        del roots_m
        # the two paths are the same function up to the rounding of the network (fp16 storage, BN folding, library kernels)
        assert agreement["root_action_agreement"] >= 0.99 or wl["config"] != 4 or N < 4096, \
            f"production path picks a different root action on {1 - agreement['root_action_agreement']:.1%} of the trees"
        if pipe.executor == "rows":
            # the searches in flight run the network on the row-block resident executor: same inputs, its own roundings
            vr, valr = h_out[0][0].to(dev), h_out[0][1].to(dev)
            agreement["rows_executor"] = {
                "root_action_agreement_with_module": float((vm.argmax(1) == vr.argmax(1)).float().mean()),
                "root_action_agreement_with_library_chain": float((vp.argmax(1) == vr.argmax(1)).float().mean()),
                "root_value_max_abs_diff_with_module": float((valm - valr).abs().max())}
            assert agreement["rows_executor"]["root_action_agreement_with_module"] >= 0.99 or wl["config"] != 4 or N < 4096, \
                "row-block executor path picks different root actions"

    env_obj, selfplay_obj = None, None
    if not args.quick:
        env_obj = bench_env(torch, dist, args, wl, env, sb, barrier, max_over_ranks, e0, e1, rank, world, dev)
        # ---- whole self-play moves, device-resident (SURVEY §8f N1/N2 rows) ----
        from hanabizero_b200.selfplay import SelfPlayEngine, SelfPlayPool
        E = max(args.in_flight, 1)      # engines (actors) per GPU, each with its own N games, on its own stream

        def timed_selfplay(engines, n_moves=5):
            pool = SelfPlayPool(engines)
            pool.reset()
            for _ in range(3):          # eager search, capture, replay
                pool.step()
            pool.synchronize()
            barrier()
            e0.record()
            for _ in range(n_moves):
                pool.step()
            pool.synchronize()
            e1.record()
            barrier()
            for eng in engines:
                eng.env.check()
            return world * len(engines) * N * n_moves / (max_over_ranks(e0.elapsed_time(e1)) * 1e-3)

        make = lambda e: SelfPlayEngine(N, wl["game"], model, cfg, seeds=np.arange(N) + 7 * N * (rank * E + e + 1), mdp=wl["mdp"],
                                        stack=args.stack, device=dev, game_offset=(rank * E + e) * N)
        engines = [make(e) for e in range(E)]
        one_moves = timed_selfplay(engines[:1])
        selfplay_moves = timed_selfplay(engines) if E > 1 else one_moves
        selfplay_obj = {"metric": "selfplay_moves_per_sec", "value": selfplay_moves, "unit": "moves/s",
                        "what": "frame stack -> representation+prediction -> Roots.prepare(Dirichlet) -> run_multi -> "
                                f"select_action -> env step with auto-reset, all on the device; {E} engines (actors) of {N} games "
                                "each, every engine on its own stream (SelfPlayPool.step)",
                        "engines": E,
                        "simulations_per_sec": selfplay_moves * (S - 1),
                        "fraction_of_search_only": selfplay_moves * (S - 1) / value,
                        "one_engine": {"value": one_moves, "simulations_per_sec": one_moves * (S - 1),
                                       "fraction_of_one_search_at_a_time": one_moves * (S - 1) / value_one}}
        del engines
    clocks = sampler.stop() if rank == 0 else None

    roof = tree_roofline(torch, args, wl, sb, model, lib) if rank == 0 else None
    net_roof = None
    if rank == 0 and args.in_flight > 1 and piped_executor == "rows" and args.amp == "torch_amp":
        net_roof = network_roofline(torch, args, wl, sb, model, lib)

    # ---- CPU baseline on the box's host cores (rank 0, N=1 only) ----------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        trees_c = wl["total"]
        reps_all = max(1, int(round(1.2e6 / max(trees_c * (S - 1), 1))))
        one = cpu_reference(min(trees_c, 1024), A, S, 1, reps=max(1, reps_all // 8), env_steps_per_core=100000, game=wl["game"],
                            pyenv_steps_per_core=2000)
        allc = cpu_reference(trees_c, A, S, cores, reps=reps_all, env_steps_per_core=100000, game=wl["game"],
                             pyenv_steps_per_core=1000)
        cpu = {"value": allc["sims_per_s"], "unit": "simulations/s", "cores": allc["cores"], "kind": allc["kind"],
               "value_1core": one["sims_per_s"],
               "env_steps_per_s": allc["env_steps_per_s"], "env_steps_per_s_1core": one["env_steps_per_s"],
               "env_python_api_steps_per_s": allc["pyenv_steps_per_s"],
               "env_python_api_steps_per_s_1core": one["pyenv_steps_per_s"],
               "env_kind": allc["env_kind"],
               "sample": (f"{trees_c} {wl['game']} trees x {S - 1} simulations x {reps_all} over {allc['tree_procs']} processes "
                          f"(and {min(trees_c, 1024)} trees x {max(1, reps_all // 8)} on 1 core): reference cytree driven like "
                          "core/mcts.py with pre-generated network outputs, no model time; env: 100000 steps/core of reference "
                          "libhanabi in C++; env_python_api: the reference's own HanabiEnv.step (rl_env.py over pyhanabi.py + "
                          "cffi), 1000 steps/core (2000 on 1 core) — what its callers pay per step")}

    if rank == 0:
        line = {
            "metric": "mcts_simulations_per_sec", "value": value, "unit": "simulations/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": wl["scaling"],
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_obj(args, wl, world),
            "setup": {"network": f"{'MuZeroNetFull' if wl['game'] == 'Hanabi-Full' else 'MuZeroNet'} random-init with re-drawn heads, "
                                 f"eval mode, BN folded, {'fp16' if args.amp == 'torch_amp' else 'fp32'} library GEMMs",
                      "model_amp": args.amp, "cuda_graph": not args.no_graph, "sharding": f"roots x{world}",
                      "searches_in_flight": max(args.in_flight, 1),
                      "gemm_sm_target": (sb.pipe.gemm_sm_target if sb.pipe is not None else 0),
                      "tree_stage_limit": (sb.pipe.stage_limit if sb.pipe is not None else 0),
                      "network_executor": ("rows" if any(getattr(w, "chain", None) is not None and w.chain._use_rows
                                                         for w in sb.mcts._ws.values()) else "library"),
                      "cuda_device_max_connections": os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS"),
                      "host_us_per_submit": (1e6 * sb.pipe.host_seconds / max(sb.pipe.submitted, 1) if sb.pipe is not None else None),
                      "what": f"`value` and `e2e` keep {max(args.in_flight, 1)} independent searches of the workload's root batch in "
                              "flight per GPU, each on its own stream (SearchPipeline: the reference's actors each own such a "
                              "batch); `one_search_at_a_time` is the same K searches back to back"},
            "e2e": {"value": e2e_value, "unit": "simulations/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "SearchPipeline.submit/wait (hanabizero_b200/mcts.py): pinned host inputs in, root statistics out, "
                           f"every search; {depth} searches in flight, each slot on its own compute stream, copies on two "
                           "copy streams",
                    "serial": {"value": e2e_serial, "api": "Roots.prepare + MCTS.run_multi + get_stats on host tensors, one "
                                                           "search at a time, a stream synchronise per search"}},
            "one_search_at_a_time": {"value": value_one, "unit": "simulations/s", "ms_per_search": ms_one / K,
                                     "us_per_simulation": 1e3 * ms_one / K / (S - 1),
                                     "what": "the same K searches issued one after the other on one stream (the latency of "
                                             "a search; `value` keeps several independent searches in flight)"},
            "us_per_simulation": 1e3 * ms_one / K / (S - 1),
            "gpu_launches": int(launches_per_search * K),
            "gpu_launches_per_search": int(launches_per_search),
            "library_gemm_launches_per_search": int(gemm_per_search),
            "launches_one_search_at_a_time": {"own": int(launches_one), "library_gemm": int(gemm_one)},
            "clocks": clocks, "roofline": roof, "network_roofline": net_roof, "cpu_baseline": cpu, "weak": weak, "plan_vs_module": agreement,
            "env": env_obj, "selfplay": selfplay_obj,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def bench_env(torch, dist, args, wl, env, sb, barrier, max_over_ranks, e0, e1, rank, world, dev):
    """Hanabi env steps/s: device-resident (CUDA graph of ten steps), host-facing (bit-packed observations through the
    double-buffered EnvPipeline; byte and float32 variants for comparison), the scalar drop-in HanabiEnv.step, the
    kernel's roofline line, and a saturated run with many more games than trees."""
    from hanabizero_b200.hanabi_env import EnvPipeline, HanabiEnv, HanabiVecEnv
    N, A, T = env.num_games, env.num_actions, args.env_steps
    legal = sb.legal
    rng = np.random.default_rng(11 + rank)
    acts_buf = torch.zeros(N, dtype=torch.int32, device=dev)

    def device_pass(e, steps, lg, buf, fused):
        """Random legal play on the device.  fused: the env kernel draws the next move itself
        (hz_envs_set_random_policy; a step is ONE launch); else three torch kernels pick it from the legal mask."""
        for _ in range(steps):
            if not fused:
                buf.copy_(torch.argmax(lg * torch.rand_like(lg), dim=1))
            _, _, lg, _, _, _ = e.step_all(buf, auto_reset=True, want_local=False)
        return lg

    def timed_graph(e, lg, buf, total_steps, per_graph=10, fused=True):
        if fused:
            e.set_random_policy(buf, seed=20 + rank)
            _, _, lg = e.observe(want_local=False)          # draw 0: the moves of the current positions
        lg = device_pass(e, 20, lg, buf, fused)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            device_pass(e, per_graph, lg, buf, fused)
        reps = max(total_steps // per_graph, 1)
        gr.replay()
        barrier()
        e0.record()
        for _ in range(reps):
            gr.replay()
        e1.record()
        barrier()
        e.set_random_policy(None)
        return world * e.num_games * reps * per_graph / (max_over_ranks(e0.elapsed_time(e1)) * 1e-3), reps * per_graph

    env_torch_policy, _ = timed_graph(env, legal, acts_buf, T, fused=False)
    env_value, steps_timed = timed_graph(env, legal, acts_buf, T)
    env.check()

    # saturated: many more games per GPU than the search has trees (the env kernel alone is latency-bound at 4096)
    sat = {}
    for games in (16384, 65536):
        big = HanabiVecEnv(games, wl["game"], np.arange(games) + 1000003 * (rank + 1), device=dev)
        _, _, lg = big.reset_all()
        v, _ = timed_graph(big, lg, torch.zeros(games, dtype=torch.int32, device=dev), max(T // 2, 20))
        big.check()
        sat[str(games)] = v
        del big

    # host-facing: actions from pinned host memory in, observation + legal mask out, every step
    T_host = max(T // 2, 20)

    # two independent half-batches: while the host reads one half's result and picks its actions, the other half's
    # copies and kernel are in flight
    G = 2 if N >= 2 else 1
    n_g = N // G
    halves = [HanabiVecEnv(n_g, wl["game"], np.arange(n_g) + 500009 * (rank * G + gi + 1), device=dev) for gi in range(G)]
    for h in halves:
        h.reset_all(observe=False)
    # host policy: a uniformly random legal move per game from the returned legal mask (hz_host_random_legal, a few
    # nanoseconds per game in C; numpy needs ~15 vectorised passes = more than the whole device step)
    rows_tmp = [torch.zeros(n_g, 4, dtype=torch.int32) for _ in range(G)]

    def timed_pipeline(fmt, zero_copy=None):
        """wait -> pick -> step, round-robin over the half-batches: while the host handles one half, the other half's
        kernel (and its PCIe traffic) is in flight."""
        pipe = EnvPipeline(halves, fmt=fmt, zero_copy=zero_copy)
        h_acts = [pipe.actions(gi) for gi in range(G)]          # the pipeline's own pinned action buffers
        shifts = np.arange(A, dtype=np.uint32)
        for gi in range(G):
            pipe.observe_now(gi)
        def one_step(gi, step):
            obs, leg = pipe.wait(gi)                      # pinned host views of the group's previous step
            if fmt == "bits":
                rows = leg                                  # meta rows [n, 4]: word 0 is the legal mask
            else:                                           # 0/1 rows -> the same mask word
                rows = rows_tmp[gi]
                rows[:, 0] = torch.from_numpy((leg.numpy().astype(np.uint32) << shifts).sum(1, dtype=np.uint32).view(np.int32))
            halves[gi].random_legal_host(rows, h_acts[gi], seed=rank, step=step)
            pipe.step(gi)

        for step in range(5):             # warm-up (the staged variants capture their graphs here)
            for gi in range(G):
                one_step(gi, step)
        barrier()
        e0.record()
        for step in range(5, 5 + T_host):     # one host thread, round-robin over the halves (threads bought nothing)
            for gi in range(G):
                one_step(gi, step)
        pipe.drain()
        e1.record()
        barrier()
        v = world * n_g * G * T_host / (max_over_ranks(e0.elapsed_time(e1)) * 1e-3)
        return v, pipe.d2h_bytes_per_step

    e2e_bits, d2h_bits = timed_pipeline("bits")
    e2e_staged, _ = timed_pipeline("bits", zero_copy=False)
    e2e_u8, d2h_u8 = timed_pipeline("u8")
    e2e_f32, d2h_f32 = timed_pipeline("f32")
    for h in halves:
        h.check()
    del halves

    # the scalar drop-in (rl_env.py API, one game): what a caller that keeps the reference's loop gets
    scalar = None
    if rank == 0:
        one = HanabiEnv({"hanabi_name": wl["game"], "seed": 1})
        _, _, lg1 = one.reset()
        n_sc = 300
        t0 = time.perf_counter()
        for _ in range(n_sc):
            _, _, _, done, _, lg1 = one.step(int(rng.choice(np.flatnonzero(np.asarray(lg1)))))
            if done:
                _, _, lg1 = one.reset()
        scalar = n_sc / (time.perf_counter() - t0)

    # roofline of the env kernel: one launch at a time, L2 flushed, float32 observations (what the network eats)
    env_roof = None
    if rank == 0:
        peak, peak_src = measured_peak()
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        evs = []
        lg = env.legal
        for _ in range(30):
            flush.fill_(1)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            acts_buf.copy_(torch.argmax(lg * torch.rand_like(lg), dim=1))
            a0.record()
            _, _, lg, _, _, _ = env.step_all(acts_buf, auto_reset=True, want_local=False)
            a1.record()
            evs.append((a0, a1))
        torch.cuda.synchronize()
        d2 = statistics.mean(a.elapsed_time(b) for a, b in evs) * 1e-3
        by = N * b_env_step(env.global_dim, A, 4)
        env_traffic, env_traffic_src = ncu_env_traffic_per_launch(N)
        env_roof = {"bound": "hbm", "kernel": "k_env<step,observe> (float32 observations)", "achieved": by / d2 / 1e9,
                    "peak": peak, "unit": "GB/s", "frac": by / d2 / 1e9 / peak, "traffic": env_traffic,
                    "traffic_source": env_traffic_src,
                    "traffic_note": "DRAM bytes with the caches as the previous step left them: the 13 MB of observations a "
                                    "launch writes stay in the 126 MB L2, so DRAM sees almost nothing",
                    "launch_us": d2 * 1e6,
                    "algorithmic_bytes_per_game": b_env_step(env.global_dim, A, 4), "peak_source": peak_src,
                    "games": N,
                    "saturated": {"games": 65536, "achieved": sat["65536"] / world * b_env_step(env.global_dim, A, 4) / 1e9,
                                  "frac": sat["65536"] / world * b_env_step(env.global_dim, A, 4) / 1e9 / peak,
                                  "what": "the same kernel in the graph-replayed loop with 65536 games per GPU: at 4096 games "
                                          "the launch lasts as long as its slowest game (a finished game re-deals ten cards "
                                          "through dependent fp64 chains), with 16x the games the SMs stay busy"}}
    return {"metric": "hanabi_env_steps_per_sec", "value": env_value, "unit": "steps/s",
            "games_per_gpu": N, "steps_timed": steps_timed,
            "includes": "random legal play on the device: ONE launch per step (step + auto-reset + float32 global observation "
                        "+ legal mask + the next random legal move, hz_envs_set_random_policy), ten steps per CUDA graph",
            "with_torch_policy": {"value": env_torch_policy,
                                  "what": "the same loop with the move picked by three torch kernels from the legal mask (what "
                                          "round 1 timed)"},
            "saturated": {"what": "the same device-resident loop with more games per GPU than the search has trees",
                          "steps_per_s_by_games_per_gpu": sat},
            "e2e": {"value": e2e_bits, "unit": "steps/s", "h2d_bytes_per_step": 4 * N, "d2h_bytes_per_step": d2h_bits,
                    "obs_format": "bits",
                    "what": "EnvPipeline (hanabizero_b200/hanabi_env.py): actions in pinned host memory in, the global "
                            "observation as a bit string (785 bits -> 100 bytes per game) + legal mask + reward/done/score out "
                            "to pinned host memory every step, the host picks the next action from the returned mask "
                            "(hz_host_random_legal); no staging copies: the kernel reads the actions from and writes the rows "
                            "to the pinned buffers itself (hz_envs_host_step, one launch + one event record per half-step); two "
                            "half-batches in flight on two streams, one host thread",
                    "bits_staged": {"value": e2e_staged, "what": "the same rows through device staging buffers: H2D copy, "
                                                                  "kernel, two D2H copies, replayed as one CUDA graph"},
                    "u8": {"value": e2e_u8, "d2h_bytes_per_step": d2h_u8},
                    "f32": {"value": e2e_f32, "d2h_bytes_per_step": d2h_f32}},
            "scalar_dropin_steps_per_s": scalar,
            "roofline": env_roof}


def measured_peak():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    if "hbm_gbs" in peaks:
        return float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


def network_roofline(torch, args, wl, sb, model, lib):
    """Tensor roofline of the network executor the in-flight searches run (k_row_chain, hz_rowchain): algorithmic
    FLOPs of one recurrent_inference (2 x in x out over the reference's Linear layers, the one-hot action columns
    included, no padding) x rows per launch / launch duration, measured live with CUDA events two ways: D launches
    in flight on D streams back to back (the regime the executor is built for: each launch holds rows/128 SMs), and
    one launch after another on one stream (a launch alone leaves most SMs idle by design)."""
    from hanabizero_b200.plan import BoundChain
    plan = model.recurrent_plan(torch.float16)
    N = wl["per_gpu"]
    probe = BoundChain(plan, N)
    if not probe.rows_supported():
        return None
    net = model
    flops_row = 0
    for m in net.modules():
        if isinstance(m, torch.nn.Linear) and not any(m is x for x in net._representation.modules()):
            flops_row += 2 * m.in_features * m.out_features
    D = max(1, int(args.in_flight))
    reps = 25
    chains = [probe] + [BoundChain(plan, N) for _ in range(D - 1)]
    for c in chains:
        c.x0.copy_((torch.rand(c.x0.shape, device=c.x0.device) * 0.5).to(c.x0.dtype))
        c.set_executor("rows")
        c.bind_state(c.state)
    streams = [torch.cuda.Stream() for _ in chains]
    graphs = []
    for c, st in zip(chains, streams):
        with torch.cuda.stream(st):
            c.run(st.cuda_stream)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            for _ in range(reps):
                c.run(torch.cuda.current_stream().cuda_stream)
        graphs.append(g)

    def timed(n_streams):
        e0 = torch.cuda.Event(enable_timing=True)
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(n_streams)]
        for st, g in list(zip(streams, graphs))[:n_streams]:
            with torch.cuda.stream(st):
                g.replay()
        torch.cuda.synchronize()
        e0.record()
        for st, g, e in list(zip(streams, graphs, ends))[:n_streams]:
            st.wait_event(e0)
            with torch.cuda.stream(st):
                g.replay(); g.replay(); e.record(st)
        torch.cuda.synchronize()
        return max(e0.elapsed_time(e) for e in ends) * 1e-3 / (2 * reps * n_streams)    # seconds per launch, aggregate

    t_flight, t_alone = timed(D), timed(1)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    src = "measured cuBLAS bf16, sustained (MEASURED_PEAKS.json)" if "bf16_tflops_sustained" in peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    fl = flops_row * N
    return {"bound": "tensor", "kernel": "k_row_chain (hz_rowchain_run): dynamics + reward/value/policy heads of one simulation, fp16 x fp16 -> fp32",
            "achieved": fl / t_flight / 1e12, "peak": peak, "unit": "TFLOP/s", "frac": fl / t_flight / 1e12 / peak,
            "peak_source": src, "launches_in_flight": D, "launch_us_aggregate": t_flight * 1e6,
            "algorithmic_flops_per_launch": fl, "algorithmic_flops_per_row": flops_row, "rows_per_launch": N,
            "ctas_per_launch": -(-N // 128),
            "alone": {"launch_us": t_alone * 1e6, "achieved": fl / t_alone / 1e12, "frac": fl / t_alone / 1e12 / peak,
                      "what": "one launch after another on one stream: rows/128 CTAs busy, the other SMs idle (they are "
                              "what the other searches in flight use)"},
            "library_chain": "seven cuBLASLt launches of the same function: see profiles/r02_rowchain.md",
            "traffic": None}


def tree_roofline(torch, args, wl, sb, model, lib, stage_limit=None):
    """Roofline of the dominant kernel of this repository — the fused tree step (hz_trees_search_step: decode +
    expand + back-propagate + min/max + traverse + hand-off) — timed live: one launch per simulation on synthetic
    network outputs, alone on the stream, L2 flushed before every launch; and the same launches back to back inside
    a CUDA graph (what the search loop sees).  The launch is the one the timed searches run: with the staging limit of
    the searches in flight (hz_search_io.stage_limit); the variant a search that runs alone uses (everything staged) is
    reported beside it."""
    own_limit = stage_limit is None
    if own_limit:
        stage_limit = sb.pipe.stage_limit if sb.pipe is not None else 0
    from hanabizero_b200 import _lib, cytree
    N, A, S, F, dev = sb.n, sb.A, sb.S, F_HIDDEN, sb.dev
    peak, peak_src = measured_peak()
    plan = model.recurrent_plan(torch.float16 if args.amp == "torch_amp" else torch.float32)
    ch = plan.chain(N)
    eb = ch.x0.element_size()
    ch.out.copy_(torch.randn_like(ch.out.float()).to(ch.out.dtype))
    roots = cytree.Roots(N, A, S, device=dev)
    roots.prepare(CONST["frac"], sb.noise, sb.zeros_r, sb.root_logits, sb.legal_i)
    mm = cytree.MinMaxStatsList(N); mm.set_delta(CONST["delta"])
    pool = torch.rand(S, N, F, device=dev).to(ch.x0.dtype)
    io = _lib.SearchIO()
    io.value_logits, io.ld_value = ch.value_logits.data_ptr(), ch.value_logits.stride(0)
    io.reward_logits, io.ld_reward = ch.reward_logits.data_ptr(), ch.reward_logits.stride(0)
    io.policy_logits, io.ld_policy = ch.policy_logits.data_ptr(), ch.policy_logits.stride(0)
    io.next_state, io.ld_state = None, 0     # as in the search loop: the dynamics GEMM writes pool[x] itself
    io.support, io.support_width, io.support_delta = plan.support.data_ptr(), plan.n_support, plan.net.support_delta
    io.elem_bytes, io.sanitize_nan = eb, 1
    io.pool, io.state_cols = pool.data_ptr(), F
    io.out_batch, io.ld_batch, io.onehot_cols = ch.x0.data_ptr(), ch.x0.stride(0), plan.OH
    io.out_ix, io.out_action = None, None
    io.minmax, io.value_delta_max = mm.tensor(dev).data_ptr(), CONST["delta"]
    io.discount, io.pb_c_base, io.pb_c_init = CONST["discount"], CONST["pb_c_base"], CONST["pb_c_init"]
    io.stage_limit = int(stage_limit)
    st = torch.cuda.current_stream().cuda_stream
    ref = _lib.C.byref(io)
    _lib.check(lib.hz_trees_search_step(roots.handle, st, 0, 1, ref))
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(S)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    depth_sum, depth_max = 0.0, []
    gen_out = torch.Generator(device=dev).manual_seed(99)
    outs = [torch.randn(ch.out.shape, device=dev, generator=gen_out).to(ch.out.dtype) for _ in range(8)]
    for x in range(1, S - 1):
        ch.out.copy_(outs[x % 8])   # fresh synthetic network outputs per simulation (realistic tree depths)
        flush.fill_(x & 1)          # evict L2: every launch starts cold
        evs[x][0].record()
        _lib.check(lib.hz_trees_search_step(roots.handle, st, x, 1, ref))
        evs[x][1].record()
        pl = roots.export(1)["path_len"].float()
        depth_sum += float(pl.mean().item()) - 1.0
        depth_max.append(int(pl.max().item()) - 1)
    torch.cuda.synchronize()
    durs = [evs[x][0].elapsed_time(evs[x][1]) * 1e-3 for x in range(1, S - 1)]
    # the same launches back to back inside a CUDA graph, no flush
    roots.prepare(CONST["frac"], sb.noise, sb.zeros_r, sb.root_logits, sb.legal_i)
    mm.clear()
    _lib.check(lib.hz_trees_search_step(roots.handle, st, 0, 1, ref))
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        st_c = torch.cuda.current_stream().cuda_stream
        for x in range(1, S - 1):
            ch.out.copy_(outs[x % 8])
            _lib.check(lib.hz_trees_search_step(roots.handle, st_c, x, 1, ref))
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0.record()
    gr.replay()
    w1.record()
    torch.cuda.synchronize()
    _lib.check(lib.hz_trees_set_progress(roots.handle, S - 2))
    gc = torch.cuda.CUDAGraph()      # the same graph without the tree launches: the copies' own cost
    with torch.cuda.graph(gc):
        for x in range(1, S - 1):
            ch.out.copy_(outs[x % 8])
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    gc.replay()
    c1.record()
    torch.cuda.synchronize()
    warm_us = (w0.elapsed_time(w1) - c0.elapsed_time(c1)) * 1e3 / (S - 2)
    D = depth_sum / len(durs)
    s_mean = statistics.mean(range(1, S - 1))
    # SURVEY §8d B_sim (tree part + the hidden-row gather in the pool's dtype) + the two support-logit rows and the
    # policy row this launch decodes.  Nothing else: the state -> pool copy of round 1 is gone from the kernel.
    per_tree = b_sim(A, D, s_mean, F * eb / 4.0) + (2 * plan.n_support + A) * eb
    bytes_launch = N * per_tree
    achieved = bytes_launch / statistics.mean(durs) / 1e9
    traffic, traffic_src = ncu_traffic_per_launch(N, stage_limit)
    solo = None
    if own_limit and stage_limit != 0:     # the variant of a search that runs alone: the whole tree staged
        full = tree_roofline(torch, args, wl, sb, model, lib, stage_limit=0)
        solo = {k: full[k] for k in ("achieved", "frac", "launch_us", "launch_us_in_graph_no_flush", "frac_in_graph_no_flush",
                                     "traffic", "traffic_source")}
        solo["what"] = "the same launch with stage_limit = 0 (a search that runs alone: as much of the tree as fits is staged)"
    return {"bound": "hbm", "kernel": "k_search_step<half,backprop,traverse> (hz_trees_search_step)",
            "stage_limit": int(stage_limit), "stage_all": solo,
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": peak_src, "launch_us": 1e6 * statistics.mean(durs), "launch_us_in_graph_no_flush": warm_us,
            "frac_in_graph_no_flush": bytes_launch / (warm_us * 1e-6) / 1e9 / peak,
            "algorithmic_bytes_per_launch": bytes_launch, "algorithmic_bytes_per_tree": per_tree,
            "mean_depth": D, "l2": "flushed before every timed launch (256 MiB write)",
            "per_sim_us_flushed": [round(1e6 * d, 1) for d in durs[::6]], "max_depth": depth_max[::6]}


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
