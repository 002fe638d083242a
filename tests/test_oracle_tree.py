"""CPU: the plain-C tree oracle (oracle/tree_oracle.c) against golden traces produced by the
unmodified reference ctree (oracle/_ref, rand()==0 shim), against the stored lock-step traces of
tests/golden/make_lockstep_traces.py and, when the reference is built, live against it."""
import numpy as np
import pytest

from helpers import (CONST, LOCKSTEP_TREE_CASES, assert_same_tree_trace, bits_equal, extreme_tree_inputs, golden_files,
                     golden_tree_inputs, load_golden, lockstep_tree_name, run_tree_lockstep, tree_inputs, tree_trace)
from oracle import loader as L


@pytest.mark.parametrize("name", golden_files("tree_"))
def test_oracle_matches_reference_golden(name):
    g = load_golden(name)
    d = golden_tree_inputs(g)
    eng = L.oracle_tree(int(g["N"]), int(g["A"]), int(g["S"]), CONST["delta"])
    run_tree_lockstep(eng, g, d)
    assert (eng.trajectories(int(g["S"])) == g["traj"]).all()
    assert (eng.path_lens() == g["plen"][-1]).all()


def test_input_generator_in_sync_with_golden():
    g = load_golden("tree_full_n8_s50.npz")
    d = tree_inputs(8, 20, 50, 1234)
    for k in d:
        assert bits_equal(d[k], g["in_" + k]), k


@pytest.mark.parametrize("N,A,S,seed,noise,mask_mode", LOCKSTEP_TREE_CASES)
def test_oracle_matches_stored_reference_trace(N, A, S, seed, noise, mask_mode):
    """The lock-step comparison below against its stored trace (tests/golden/make_lockstep_traces.py): root priors,
    every simulation's traverse outputs and root statistics, and every expanded node, bit-exact."""
    d = tree_inputs(N, A, S, seed, mask_mode)
    assert_same_tree_trace(tree_trace(L.oracle_tree(N, A, S), d, S, noise),
                           load_golden(lockstep_tree_name(N, A, S, seed, noise, mask_mode)))


@pytest.mark.skipif(not L.have_ref(), reason="oracle/_ref not built (no reference sources at build time)")
@pytest.mark.parametrize("N,A,S,seed,noise,mask_mode", LOCKSTEP_TREE_CASES)
def test_oracle_matches_live_reference(N, A, S, seed, noise, mask_mode):
    d = tree_inputs(N, A, S, seed, mask_mode)
    assert_same_tree_trace(tree_trace(L.oracle_tree(N, A, S), d, S, noise), tree_trace(L.ref_tree(N, A, S), d, S, noise))


def test_nan_and_extreme_inputs_match_stored_reference_trace():
    """NaN logits at the root (not sanitised by the reference), huge/tiny logits, NaN values: traverse outputs of every
    simulation and the final root statistics against the stored trace."""
    N, A, S, d = extreme_tree_inputs()
    assert_same_tree_trace(tree_trace(L.oracle_tree(N, A, S), d, S), load_golden("lockstep_tree_extreme.npz"),
                           per_step_stats=False, expanded=False)


@pytest.mark.skipif(not L.have_ref(), reason="oracle/_ref not built")
def test_nan_and_extreme_inputs_match_reference():
    """The same inputs live against the reference."""
    N, A, S, d = extreme_tree_inputs()
    assert_same_tree_trace(tree_trace(L.oracle_tree(N, A, S), d, S), tree_trace(L.ref_tree(N, A, S), d, S),
                           per_step_stats=False, expanded=False)


def test_random_tie_mode_is_uniform_like_the_stock_reference():
    """Tie mode 1 of the oracle (the counter-based draw the CUDA path uses) against the reference's stock build
    (rand() % ties, clock-seeded): with the reference's zero-initialised heads every select is an A-way tie, so the
    first action of a search is uniform over the actions for both — and never 'always action 0'."""
    from helpers import tree_inputs
    N, A, S = 4000, 20, 3
    d = tree_inputs(N, A, S, 5)
    for k in ("logits", "sim_logits", "sim_value", "sim_reward", "reward"):
        d[k][:] = 0.0
    d["mask"][:] = 1
    counts = {}
    engines = {"oracle": L.oracle_tree(N, A, S)}
    engines["oracle"].set_tie(1, 2024, 0)
    if L.have_ref():
        engines["reference"] = L.ref_tree(N, A, S, deterministic=False)
    for name, e in engines.items():
        e.prepare(0.25, None, d["reward"], d["logits"], d["mask"])
        la = e.traverse(19652, 1.25, 0.999)[2]
        counts[name] = np.bincount(la, minlength=A)
    for name, c in counts.items():
        chi2 = ((c - N / A) ** 2 / (N / A)).sum()
        assert chi2 < 60.0, f"{name}: first actions not uniform over {A}-way ties (chi2 {chi2:.1f}, 19 dof): {c}"
