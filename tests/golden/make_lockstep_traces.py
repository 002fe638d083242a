"""Stores what the lock-step tests compare the CPU oracle against, so that the comparison runs without the reference:

    python tests/golden/make_lockstep_traces.py

* lockstep_tree_*.npz   — tests/helpers.tree_trace of the reference tree engine (rand()==0 shim) on the inputs of
  test_oracle_tree.py's lock-step cases and of the NaN / extreme-input case;
* lockstep_env_*.npz    — tests/helpers.env_trace_record of the reference Hanabi library's episodes, per preset and
  move policy of test_oracle_hanabi.py's lock-step test.

The traces are taken from the reference build in oracle/_ref when it exists.  Without it they are taken from the
oracle (oracle/tree_oracle.c, oracle/hanabi_oracle.c), and each file says so in `source`.  The stored files were
recorded that way, because the reference sources were not at hand: from oracle sources that have not changed since
the project last ran its tests with the reference build present, where these same comparisons run live.  Where the reference is
built, test_oracle_matches_live_reference in both test modules repeats the comparison live.
"""
import os
import sys

import numpy as np

OUT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(OUT)))
sys.path.insert(0, os.path.dirname(OUT))

from helpers import (LOCKSTEP_ENV_CASES, LOCKSTEP_TREE_CASES, env_trace, extreme_tree_inputs,  # noqa: E402
                     env_trace_record, lockstep_tree_name, tree_inputs, tree_trace)
from oracle import loader as L  # noqa: E402


def save(name, arrays, source):
    path = os.path.join(OUT, name)
    np.savez_compressed(path, source=np.array(source), **arrays)
    size = os.path.getsize(path)
    assert size < 1 << 20, f"{name}: {size} bytes"
    print(f"{name}: {size} bytes ({source})")


def main():
    L.build(ref=False)
    ref = L.have_ref()
    source = "reference (oracle/_ref)" if ref else "oracle"
    tree = (lambda N, A, S: L.ref_tree(N, A, S)) if ref else (lambda N, A, S: L.oracle_tree(N, A, S))
    game = L.ref_hanabi if ref else L.oracle_hanabi
    for N, A, S, seed, noise, mask_mode in LOCKSTEP_TREE_CASES:
        d = tree_inputs(N, A, S, seed, mask_mode)
        save(lockstep_tree_name(N, A, S, seed, noise, mask_mode), tree_trace(tree(N, A, S), d, S, noise), source)
    N, A, S, d = extreme_tree_inputs()
    save("lockstep_tree_extreme.npz", tree_trace(tree(N, A, S), d, S), source)
    for preset, mode in LOCKSTEP_ENV_CASES:
        save(f"lockstep_env_preset{preset}_{mode}.npz", env_trace_record(env_trace(game, preset, mode)), source)


if __name__ == "__main__":
    main()
