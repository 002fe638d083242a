"""CPU: the recorded fast path's entry points (hz_traj_record_u8, hz_envs_step_observe_u8_terminal) reject bad
arguments before anything is launched, their ctypes types follow include/hzb200.h, and SelfPlayEngine(record="ring")
refuses a model it cannot run on the byte frame ring (no GPU here: a launch would fail differently and count)."""
import ctypes
import os
import re

import pytest

from helpers import ROOT

N, D, A, S, L, B = 5, 173, 11, 4, 16, 2
BUF = 0x10000                       # 16-byte aligned stand-in: the checks reject the call before any access


def _view(**kw):
    from hanabizero_b200 import _lib
    v = _lib.TrajView()
    for name in ("obs", "legal", "action", "reward", "visits", "root_value", "len", "bank", "finished", "overflow"):
        setattr(v, name, BUF)
    v.num, v.obs_dim, v.actions, v.stack, v.max_len, v.banks = N, D, A, S, L, B
    for k, x in kw.items():
        setattr(v, k, x)
    return v


def _record(view=None, **kw):
    from hanabizero_b200 import _lib
    args = dict(actions=BUF, reward=BUF, visits=BUF, root_values=BUF, done=BUF, next_obs=BUF, ld_next=176,
                next_legal=BUF, term_obs=BUF, ld_term=176, term_legal=BUF, active=None)
    args.update(kw)
    v = _view() if view is None else view
    return _lib.load().hz_traj_record_u8(None, ctypes.byref(v), *args.values())


RECORD_BAD = {
    "NULL view obs": dict(view=dict(obs=None)),
    "NULL view overflow": dict(view=dict(overflow=None)),
    "view num 0": dict(view=dict(num=0)),
    "view obs_dim 0": dict(view=dict(obs_dim=0)),
    "view actions 33": dict(view=dict(actions=33)),
    "view banks 1": dict(view=dict(banks=1)),
    "view max_len 0": dict(view=dict(max_len=0)),
    "view stack 0": dict(view=dict(stack=0)),
    **{f"NULL {k}": {k: None} for k in ("actions", "reward", "visits", "root_values", "done", "next_obs", "next_legal",
                                         "term_obs", "term_legal")},
    "ld_next < obs_dim": dict(ld_next=D - 1),
    "ld_term < obs_dim": dict(ld_term=D - 1),
}


@pytest.mark.parametrize("case", list(RECORD_BAD))
def test_traj_record_u8_rejects_bad_arguments_without_a_launch(case):
    from hanabizero_b200 import _lib
    lib = _lib.load()
    kw = dict(RECORD_BAD[case])
    view = _view(**kw.pop("view")) if "view" in kw else None
    before = lib.hz_launch_count()
    assert _record(view, **kw) == _lib.HZ_ERR_ARG
    assert b"hz_traj_record_u8" in lib.hz_last_error()
    assert lib.hz_launch_count() == before


def test_traj_record_u8_rejects_a_missing_view():
    from hanabizero_b200 import _lib
    lib = _lib.load()
    before = lib.hz_launch_count()
    assert lib.hz_traj_record_u8(None, None, BUF, BUF, BUF, BUF, BUF, BUF, 176, BUF, BUF, 176, BUF, None) == _lib.HZ_ERR_ARG
    assert lib.hz_launch_count() == before


def test_terminal_step_rejects_a_null_handle():
    from hanabizero_b200 import _lib
    lib = _lib.load()
    before = lib.hz_launch_count()
    assert lib.hz_envs_step_observe_u8_terminal(None, None, BUF, None, BUF, BUF, BUF, BUF, 800, None, 0, BUF, BUF, 800,
                                                BUF) == _lib.HZ_ERR_ARG
    assert b"hz_envs_step_observe_u8_terminal" in lib.hz_last_error()
    assert lib.hz_launch_count() == before


def test_ring_recording_needs_an_initial_plan():
    from hanabizero_b200.mcts import SearchConfig
    from hanabizero_b200.selfplay import SelfPlayEngine

    class NoPlan:                   # a model with only the module's root inference
        def initial_inference_device(self, obs):
            raise AssertionError("not reached")

    with pytest.raises(ValueError, match="initial_plan"):
        SelfPlayEngine(4, "Hanabi-Full", NoPlan(), SearchConfig(num_simulations=4), record="ring")
    with pytest.raises(ValueError, match="record"):
        SelfPlayEngine(4, "Hanabi-Full", NoPlan(), SearchConfig(num_simulations=4), record="rings")


def _header_params(name):
    text = open(os.path.join(ROOT, "include", "hzb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    m = re.search(r"\bint\s+" + name + r"\s*\(([^)]*)\)\s*;", text)
    assert m, name
    return [" ".join(p.split()) for p in m.group(1).split(",")]


def _ctype(param):
    if "*" in param:
        return ctypes.c_void_p
    kind = param.rsplit(" ", 1)[0].replace("const ", "")
    return {"int": ctypes.c_int, "int64_t": ctypes.c_int64, "float": ctypes.c_float, "double": ctypes.c_double,
            "uint64_t": ctypes.c_uint64, "uint32_t": ctypes.c_uint32}[kind]


@pytest.mark.parametrize("name", ["hz_traj_record_u8", "hz_envs_step_observe_u8_terminal"])
def test_binding_types_follow_the_header(name):
    from hanabizero_b200 import _lib
    res, args = _lib.SIGNATURES[name]
    assert res is ctypes.c_int
    assert args == [_ctype(p) for p in _header_params(name)]
