"""CPU: argument checks of hz_rowchain_create_small, the Hanabi-Small entry of the row-block resident executor.  Every
case fails with HZ_ERR_ARG before a device is touched (no GPU here), so a wrong shape or pointer is an error, never a
kernel running with the wrong layout."""
import ctypes

import pytest

SMALL = dict(ld_w1=528, state_cols=512, head_cols=128, onehot_cols=16, logit_cols=64)
FULL_ONLY = ("wb2", "bb2", "wa2", "ba2")
BUF = ctypes.c_void_p(0x1000)


def _weights(**over):
    from hanabizero_b200 import _lib
    w = _lib.RowChainWeights()
    for f, _ in _lib.RowChainWeights._fields_:
        if f not in SMALL and f not in FULL_ONLY:
            setattr(w, f, 0x1000)
    for f, v in {**SMALL, **over}.items():
        setattr(w, f, v)
    return w


def _create(w, rows=128, x0=BUF, ld_x0=528, state=BUF, out=BUF):
    from hanabizero_b200 import _lib
    lib = _lib.load()
    h = ctypes.c_void_p()
    status = lib.hz_rowchain_create_small(ctypes.byref(h), 0, None if w is None else ctypes.byref(w), rows, x0, ld_x0,
                                          state, out)
    return status, lib.hz_last_error()


def _arg_error(**kw):
    from hanabizero_b200 import _lib
    status, msg = _create(**kw)
    assert status == _lib.HZ_ERR_ARG, (status, msg)
    assert b"hz_rowchain_create_small" in msg
    return msg


def test_missing_handle_weights_or_buffers():
    _arg_error(w=None)
    _arg_error(w=_weights(), rows=0)
    _arg_error(w=_weights(), x0=None)
    _arg_error(w=_weights(), state=None)
    _arg_error(w=_weights(), out=None)


def test_full_shapes_are_rejected():
    msg = _arg_error(w=_weights(head_cols=256, onehot_cols=32, logit_cols=208, ld_w1=544), ld_x0=544)
    assert b"heads 128" in msg
    _arg_error(w=_weights(head_cols=256))


@pytest.mark.parametrize("cols", [32, 0, 11])
def test_one_hot_width_other_than_16(cols):
    _arg_error(w=_weights(onehot_cols=cols, ld_w1=544), ld_x0=544)


@pytest.mark.parametrize("cols", [0, 16, 48, 51, 80, 208, 256])
def test_logit_width_other_than_64(cols):
    _arg_error(w=_weights(logit_cols=cols))


def test_strides_too_narrow_or_unaligned():
    _arg_error(w=_weights(), ld_x0=512)      # no room for the one-hot columns
    _arg_error(w=_weights(), ld_x0=532)      # rows not 16-byte aligned
    _arg_error(w=_weights(ld_w1=512))
    _arg_error(w=_weights(ld_w1=530))


@pytest.mark.parametrize("field", FULL_ONLY)
def test_full_only_pointers_must_be_null(field):
    msg = _arg_error(w=_weights(**{field: 0x1000}))
    assert b"NULL" in msg


@pytest.mark.parametrize("field", ["w1", "w1a_t", "b1", "w2", "b2", "w3", "b3", "wh1", "bh1", "wb3", "bb3"])
def test_null_and_misaligned_weight_pointers(field):
    assert b"pointer" in _arg_error(w=_weights(**{field: 0}))
    assert b"pointer" in _arg_error(w=_weights(**{field: 0x1008}))


def test_misaligned_buffers():
    odd = ctypes.c_void_p(0x1008)
    for kw in (dict(x0=odd), dict(state=odd), dict(out=odd)):
        assert b"pointer" in _arg_error(w=_weights(), **kw)


def test_full_entry_still_rejects_small_shapes():
    """The two entry points do not overlap: Hanabi-Small shapes are an argument error of hz_rowchain_create."""
    from hanabizero_b200 import _lib
    lib = _lib.load()
    h = ctypes.c_void_p()
    w = _weights()
    launches = lib.hz_launch_count()          # (GPU tests earlier in the same process have launched kernels)
    assert lib.hz_rowchain_create(ctypes.byref(h), 0, ctypes.byref(w), 128, BUF, 528, BUF, BUF) == _lib.HZ_ERR_ARG
    assert lib.hz_launch_count() == launches


def test_auto_executor_follows_the_measured_crossover():
    """executor="auto" for searches in flight: Hanabi-Full always takes the row executor; Hanabi-Small only from 48
    row blocks in flight, the crossover measured on B200 (32 blocks: library faster, 48: rows faster)."""
    from hanabizero_b200.mcts import network_executor_for

    class Net:
        def __init__(self, full):
            self.full = full

    full, small = Net(True), Net(False)
    for n, d in ((4096, 1), (16, 1), (512, 1)):
        assert network_executor_for(full, n, d) == network_executor_for(small, n, d) == "library"
    for n, d in ((16, 7), (512, 4), (512, 8), (1024, 4), (4096, 2)):
        assert network_executor_for(full, n, d) == "rows"
    for n, d in ((16, 7), (512, 4), (512, 8), (1024, 4), (1000, 5), (1900, 3)):
        assert network_executor_for(small, n, d) == "library", (n, d)
    for n, d in ((768, 8), (512, 12), (512, 20), (1024, 8), (4096, 8), (2048, 3), (4096, 12)):
        assert network_executor_for(small, n, d) == "rows", (n, d)
