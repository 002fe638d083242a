"""CPU: the plain-C Hanabi oracle (oracle/hanabi_oracle.c) against golden episodes produced by the
reference's own Python HanabiEnv, against the stored lock-step episodes of tests/golden/make_lockstep_traces.py and,
when the reference is built, live against the compiled reference library."""
import numpy as np
import pytest

from helpers import (assert_same_env_trace, env_trace, env_trace_record, golden_files, load_golden,
                     unpack_env_golden)
from oracle import loader as L


@pytest.mark.parametrize("name", golden_files("env_"))
def test_oracle_replays_reference_python_env(name):
    g = load_golden(name)
    glob_, loc = unpack_env_golden(g)
    env = L.oracle_hanabi(int(g["preset"]), int(g["seed"]))
    assert env.global_dim == int(g["glob_dim"]) and env.local_dim == int(g["loc_dim"])
    starts = set(int(s) for s in g["ep_start"])
    for t in range(len(g["action"])):
        if t in starts:
            go, lo, legal = env.reset()
            r, d, sc = 0, False, 0
        else:
            go, lo, legal, r, d, sc = env.step(int(g["action"][t]))
        assert (go == glob_[t]).all(), f"global obs differs at step {t}"
        assert (lo == loc[t]).all(), f"local obs differs at step {t}"
        assert (legal == g["legal"][t]).all(), f"legal mask differs at step {t}"
        assert (r, int(d), sc) == (int(g["reward"][t]), int(g["done"][t]), int(g["score"][t])), t


def test_shapes():
    full, small = L.oracle_hanabi(0, 0), L.oracle_hanabi(1, 0)
    assert (full.enc_len, full.own_len, full.actions, full.local_dim, full.global_dim) == (658, 125, 20, 660, 785)
    assert (small.enc_len, small.own_len, small.actions, small.local_dim, small.global_dim) == (171, 20, 11, 173, 193)


def test_illegal_action_rejected():
    env = L.oracle_hanabi(0, 0)
    _, _, legal = env.reset()
    bad = int(np.flatnonzero(legal == 0)[0])
    with pytest.raises(ValueError):
        env.step(bad)


@pytest.mark.parametrize("preset", [0, 1])
@pytest.mark.parametrize("mode", ["random", "noplay", "smart"])
def test_oracle_matches_stored_reference_episodes(preset, mode):
    """The lock-step comparison below against its stored record (tests/golden/make_lockstep_traces.py): 6 seeds x 4
    episodes on one game object per seed, observations, legal masks, state dumps, rewards and scores row by row."""
    assert_same_env_trace(env_trace_record(env_trace(L.oracle_hanabi, preset, mode)),
                          load_golden(f"lockstep_env_preset{preset}_{mode}.npz"))


@pytest.mark.skipif(not L.have_ref(), reason="oracle/_ref not built")
@pytest.mark.parametrize("preset", [0, 1])
@pytest.mark.parametrize("mode", ["random", "noplay", "smart"])
def test_oracle_matches_live_reference(preset, mode):
    assert_same_env_trace(env_trace_record(env_trace(L.oracle_hanabi, preset, mode)),
                          env_trace_record(env_trace(L.ref_hanabi, preset, mode)))
