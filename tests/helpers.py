"""Shared test helpers (test infrastructure)."""
import glob
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
CONST = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.999, delta=0.006, frac=0.25)


def golden_files(prefix):
    return sorted(os.path.basename(p) for p in glob.glob(os.path.join(GOLDEN, prefix + "*.npz")))


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def tree_inputs(N, A, S, seed, mask_mode="random"):
    """Identical to tests/golden/make_golden.py:tree_inputs (kept in sync by test_oracle_tree)."""
    rng = np.random.default_rng(seed)
    d = dict(
        logits=rng.standard_normal((N, A)).astype(np.float32),
        noise=rng.dirichlet([0.3] * A, N).astype(np.float32),
        reward=rng.standard_normal(N).astype(np.float32),
        sim_reward=rng.standard_normal((S - 1, N)).astype(np.float32),
        sim_value=rng.standard_normal((S - 1, N)).astype(np.float32),
        sim_logits=rng.standard_normal((S - 1, N, A)).astype(np.float32))
    mask = (rng.random((N, A)) < 0.6).astype(np.int32)
    mask[np.arange(N), rng.integers(0, A, N)] = 1
    if mask_mode == "zero_rows":
        mask[::3] = 0
        d["noise"] = d["noise"] * mask
    d["mask"] = mask
    return d


def golden_tree_inputs(g):
    if "in_logits" in g.files:
        return {k[3:]: g[k] for k in g.files if k.startswith("in_")}
    return tree_inputs(int(g["N"]), int(g["A"]), int(g["S"]), int(g["seed"]), str(g["mask_mode"]))


def bits_equal(a, b):
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    if a.dtype == np.float32:
        # NaN payload/sign is not part of the contract (x86 SSE yields 0xffc00000, the GPU 0x7fffffff)
        both_nan = np.isnan(a) & np.isnan(b)
        return a.shape == b.shape and bool(((a.view(np.uint32) == b.view(np.uint32)) | both_nan).all())
    return a.shape == b.shape and bool((a == b).all())


def run_tree_lockstep(engine, g, d, check_each_sim=True):
    """Drive `engine` (oracle.loader.TreeEngine-like API) through the golden trace `g`."""
    S = int(g["S"])
    engine.prepare(CONST["frac"], d["noise"] if int(g["noise"]) else None, d["reward"], d["logits"],
                   d["mask"])
    assert bits_equal(engine.root_priors(), g["priors"]), "root priors differ"
    for s in range(S - 1):
        ix, iy, la = engine.traverse(CONST["pb_c_base"], CONST["pb_c_init"], CONST["discount"])
        if check_each_sim:
            assert (ix == g["ix"][s]).all(), f"hidden_state_index_x differs at simulation {s}"
            assert (iy == g["iy"][s]).all(), f"hidden_state_index_y differs at simulation {s}"
            assert (la == g["la"][s]).all(), f"last_action differs at simulation {s}"
        engine.backprop(s + 1, CONST["discount"], d["sim_reward"][s], d["sim_value"][s],
                        d["sim_logits"][s])
    visits, values, minmax = engine.stats()
    assert (visits == g["visits"]).all(), "visit counts differ"
    assert (visits.argmax(1) == g["visits"].argmax(1)).all(), "selected actions differ"
    np.testing.assert_allclose(values, g["values"], rtol=1e-5, atol=0)   # north-star tolerance
    np.testing.assert_allclose(minmax, g["minmax"], rtol=1e-5, atol=0)
    assert bits_equal(values, g["values"]) and bits_equal(minmax, g["minmax"]), \
        "within 1e-5 but not bit-exact (expected bit-exact)"
    return visits, values, minmax


def env_policy(mode, rng, hand_size, legal, playable_slots):
    """Identical to tests/golden/make_golden.py:policy."""
    ids = np.flatnonzero(legal)
    h = hand_size
    nonplay = [a for a in ids if not (h <= a < 2 * h)]
    if mode == "random":
        return int(ids[rng.integers(len(ids))])
    if mode == "smart" and playable_slots and rng.random() < 0.9:
        return h + int(playable_slots[rng.integers(len(playable_slots))])
    if nonplay:
        return int(nonplay[rng.integers(len(nonplay))])
    return int(ids[rng.integers(len(ids))])


def playable_from_dump(dump, colors, ranks, hand_size):
    """Playable slots of the current player from the state-dump layout of oracle/hanabi_oracle.c."""
    cur = int(dump[0])
    fw = dump[5:5 + colors]
    off = 5 + colors + 2 * colors * ranks + cur * (1 + 5 * hand_size)
    n = int(dump[off])
    return [k for k in range(n) if dump[off + 1 + 5 * k] % ranks == fw[dump[off + 1 + 5 * k] // ranks]]


def unpack_env_golden(g):
    glob_ = np.unpackbits(g["glob_bits"], axis=1)[:, :int(g["glob_dim"])]
    loc = np.unpackbits(g["loc_bits"], axis=1)[:, :int(g["loc_dim"])]
    return glob_, loc


# ---- lock-step traces of the oracle against the reference (tests/golden/make_lockstep_traces.py stores them) ----
LOCKSTEP_TREE_CASES = [(32, 20, 50, 11, True, "random"), (16, 11, 50, 12, True, "random"),
                       (8, 20, 120, 13, False, "random"), (9, 20, 40, 14, True, "zero_rows"),
                       (1, 20, 50, 15, True, "random")]
LOCKSTEP_ENV_CASES = [(preset, mode) for mode in ("random", "noplay", "smart") for preset in (0, 1)]


def lockstep_tree_name(N, A, S, seed, noise, mask_mode):
    return f"lockstep_tree_n{N}_a{A}_s{S}_seed{seed}{'' if noise else '_nonoise'}_{mask_mode}.npz"


def extreme_tree_inputs():
    """N, A, S and inputs with NaN logits at a root (not sanitised by the reference), huge/tiny logits, NaN values."""
    N, A, S = 6, 20, 12
    d = tree_inputs(N, A, S, 3)
    d["logits"][0, 3] = np.nan
    d["logits"][1, :] = -200.0
    d["logits"][1, 5] = 50.0
    d["logits"][2, :] = 1e30
    d["sim_value"][2, 3] = np.nan
    d["sim_reward"][4, 4] = np.inf
    d["mask"][5, :] = 1
    return N, A, S, d


def tree_trace(engine, d, S, noise=True):
    """One tree engine (oracle.loader.TreeEngine API) driven through `d`: root priors, then per simulation the
    traverse outputs and the root statistics after back-propagation, then every tree's expanded nodes."""
    engine.prepare(CONST["frac"], d["noise"] if noise else None, d["reward"], d["logits"], d["mask"])
    t = {"priors": engine.root_priors()}
    steps = []
    for s in range(S - 1):
        out = engine.traverse(CONST["pb_c_base"], CONST["pb_c_init"], CONST["discount"])
        engine.backprop(s + 1, CONST["discount"], d["sim_reward"][s], d["sim_value"][s], d["sim_logits"][s])
        steps.append(tuple(out) + tuple(engine.stats()))
    for i, k in enumerate(("ix", "iy", "la", "visits", "values", "minmax")):
        t[k] = np.stack([st[i] for st in steps])
    ex = [engine.expanded_stats(i, S + 1) for i in range(engine.num)]
    t["ex_n"] = np.array([len(e[0]) for e in ex], np.int32)
    for j, k in enumerate(("ex_reward", "ex_value_sum", "ex_visits")):
        t[k] = np.zeros((engine.num, S + 1), ex[0][j].dtype)
        for i, e in enumerate(ex):
            t[k][i, :len(e[j])] = e[j]
    return t


def assert_same_tree_trace(a, b, per_step_stats=True, expanded=True):
    """Bit-exact agreement of two tree_trace records (per_step_stats=False: the root statistics after the last
    simulation only; expanded=False: without the expanded nodes)."""
    assert bits_equal(a["priors"], b["priors"]), "root priors"
    for k in ("ix", "iy", "la"):
        bad = np.flatnonzero((a[k] != b[k]).any(1))
        assert not len(bad), f"{k} differs first at simulation {bad[:1]}"
    for k in ("visits", "values", "minmax"):
        if per_step_stats:
            bad = [s for s in range(len(a[k])) if not bits_equal(a[k][s], b[k][s])]
            assert not bad, f"{k} differs first at simulation {bad[0]}"
        else:
            assert bits_equal(a[k][-1], b[k][-1]), k
    if expanded:
        for k in ("ex_n", "ex_reward", "ex_value_sum", "ex_visits"):
            assert bits_equal(a[k], b[k]), k


def env_trace(make, preset, mode, seeds=6, episodes=4):
    """Episodes of one Hanabi engine (oracle.loader.HanabiGameCPU API, `make(preset, seed)`): the same game object
    per seed over `episodes` resets (the mt19937 stream persists across resets), moves picked by env_policy from the
    engine's own state dump.  One row per reset (kind 0) or step (kind 1); `dump` is the state before a step."""
    rows = {k: [] for k in ("kind", "action", "glob", "loc", "legal", "rds", "dump", "dump_n")}

    def add(kind, action, obs, rds, dump):
        for k, v in zip(("kind", "action", "glob", "loc", "legal", "rds"), (kind, action) + tuple(obs) + (rds,)):
            rows[k].append(v)
        rows["dump_n"].append(len(dump))
        rows["dump"].append(np.pad(dump, (0, 256 - len(dump)), constant_values=-1))

    for seed in range(seeds):
        rng = np.random.default_rng(17 * seed + preset)
        g = make(preset, seed)
        for _ in range(episodes):
            a = g.reset()
            add(0, -1, a, (0, 0, 0), np.zeros(0, np.int32))
            done = False
            while not done:
                dump = g.dump()
                act = env_policy(mode, rng, g.hand_size, a[2], playable_from_dump(dump, g.colors, g.ranks, g.hand_size))
                a = g.step(act)
                add(1, act, a[:3], a[3:], dump)
                done = a[4]
    return {k: np.asarray(v, np.int32) for k, v in rows.items()}


def env_trace_record(t):
    """env_trace -> what is stored and compared: the episode structure, moves, reward/done/score and dump lengths in
    full, and per row one 64-bit digest of the global and local observations, the legal mask and the state dump."""
    import hashlib
    rows = np.concatenate([t[k] for k in ("glob", "loc", "legal", "dump")], axis=1).astype(np.int32)
    digest = [np.frombuffer(hashlib.blake2b(r.tobytes(), digest_size=8).digest(), np.uint64)[0] for r in rows]
    out = {k: t[k] for k in ("kind", "action", "rds", "dump_n")}
    out["row_digest"] = np.array(digest, np.uint64)
    return out


def assert_same_env_trace(a, b):
    """Two env_trace_record records agree row by row."""
    n = min(len(a["kind"]), len(b["kind"]))
    for k in ("kind", "action", "rds", "dump_n", "row_digest"):
        bad = np.flatnonzero((a[k][:n] != b[k][:n]).reshape(n, -1).any(1))
        assert not len(bad), f"{k} differs first at row {bad[0]}"
    assert len(a["kind"]) == len(b["kind"]), "episode lengths"
    assert (a["kind"] == 1).sum() > 100


class RefGameHistory:
    """The fields of core/game.py:49-215 that self-play writes, as the reference writes them (test-side port)."""

    def __init__(self, stack):
        self.stack = stack

    def init(self, init_observations, init_legal_action):            # game.py:73-93
        assert len(init_observations) == self.stack
        self.child_visits, self.root_values, self.actions, self.rewards = [], [], [], []
        self.obs_history = [np.array(o, copy=True) for o in init_observations]
        self.legal_actions = [init_legal_action]

    def store_search_stats(self, visit_counts, root_value):          # game.py:189-204 (idx is None)
        sum_visits = sum(visit_counts)
        self.child_visits.append([visit_count / sum_visits for visit_count in visit_counts])
        self.root_values.append(root_value)

    def append(self, action, obs, reward, legal_action):             # game.py:143-148
        self.actions.append(action)
        self.obs_history.append(obs)
        self.rewards.append(reward)
        self.legal_actions.append(legal_action)

    def game_over(self):                                             # game.py:176-187
        self.rewards = np.array(self.rewards)
        self.obs_history = np.array(self.obs_history)
        self.actions = np.array(self.actions)
        self.child_visits = np.array(self.child_visits)
        self.root_values = np.array(self.root_values)
        self.legal_actions = np.array(self.legal_actions)

    def put(self):                                                   # selfplay_worker.py:29-39
        prev_r = self.rewards[0]
        for step_id in range(1, len(self.rewards)):
            cur_r = self.rewards[step_id] + prev_r
            prev_r = self.rewards[step_id]
            self.rewards[step_id] = cur_r



def ref_select_action(visit_counts, temperature, deterministic, legal_actions, u):
    """core/utils.py:280-295 with np.random.choice replaced by its own algorithm for a given uniform u."""
    visit_counts = list(visit_counts)
    for i in range(len(legal_actions)):
        if legal_actions[i] == 0 and visit_counts[i] >= 1:
            visit_counts[i] = 0
    probs = [float(v) ** (1 / temperature) for v in visit_counts]
    total = sum(probs)
    probs = [x / total for x in probs]
    if deterministic:
        action = int(np.argmax(visit_counts))
    else:
        cdf = np.cumsum(np.asarray(probs, np.float64))
        cdf /= cdf[-1]
        action = int(np.searchsorted(cdf, u, side="right"))
    pk = np.asarray(probs, np.float64)
    pk = pk / pk.sum()
    ent = float(-(pk[pk > 0] * np.log(pk[pk > 0])).sum() / np.log(2))
    return action, ent, visit_counts


def unpack_traj_golden(g):
    """-> (per-step observations [T, D] uint8, list of per-episode dicts in GameHistory.save_file's layout)."""
    D, stack = int(g["obs_dim"]), int(g["stack"])
    obs = np.unpackbits(g["obs_bits"], axis=1)[:, :D]
    out_o = np.unpackbits(g["out_o_bits"], axis=1)[:, :D]
    eps, s, so, sl = [], 0, 0, 0
    for n in g["ep_len"]:
        n = int(n)
        eps.append(dict(vis=g["out_vis"][s:s + n], root=g["out_root"][s:s + n], a=g["out_a"][s:s + n],
                        r=g["out_r"][s:s + n], o=out_o[so:so + stack + n], la=g["out_la"][sl:sl + n + 1]))
        s, so, sl = s + n, so + stack + n, sl + n + 1
    return obs, eps
