"""CPU: argument checks of the byte frame ring (hz_ring_gather / hz_ring_refill, hanabizero_b200/csrc/hz_selfplay.cu).
Both kernels move 16 bytes per lane and step, so every size they take must be a multiple of 16 and every pointer
16-byte aligned; a slot index outside the ring would read or write another game's frames.  Each such call must fail
with HZ_ERR_ARG before anything is launched (no GPU here: a launch would fail differently and count)."""
import pytest

RING, OUT = 0x10000, 0x20000          # 16-byte aligned stand-ins: the checks reject the call before any access
N, S, DP = 5, 4, 208


def _gather(head=0, ring=RING, out=OUT, ld_out=S * DP, frame_stride=DP, num=N, stack=S, padded_dim=DP, elem_bytes=2):
    from hanabizero_b200 import _lib
    return _lib.load().hz_ring_gather(None, ring, head, out, ld_out, frame_stride, num, stack, padded_dim, elem_bytes)


def _refill(src_slot=0, ring=RING, done=None, num=N, stack=S, padded_dim=DP):
    from hanabizero_b200 import _lib
    return _lib.load().hz_ring_refill(None, ring, src_slot, done, num, stack, padded_dim)


GATHER_BAD = {
    "head -1": dict(head=-1),
    "head == stack": dict(head=S),
    "head past a stack of 1": dict(head=1, stack=1, ld_out=DP),
    "padded_dim 200": dict(padded_dim=200, frame_stride=208),
    "padded_dim 0": dict(padded_dim=0),
    "frame_stride 216": dict(frame_stride=216, ld_out=S * 216),
    "frame_stride < padded_dim": dict(frame_stride=192, ld_out=S * 192),
    "ld_out < stack * frame_stride": dict(ld_out=S * DP - 16),
    "ld_out 8 past a multiple of 16": dict(ld_out=S * DP + 8),
    "ring + 8": dict(ring=RING + 8),
    "ring + 1": dict(ring=RING + 1),
    "out + 8": dict(out=OUT + 8),
    "out + 4": dict(out=OUT + 4),
    "elem_bytes 3": dict(elem_bytes=3),
    "elem_bytes 1": dict(elem_bytes=1),
    "NULL ring": dict(ring=None),
    "NULL out": dict(out=None),
    "num 0": dict(num=0),
    "stack 0": dict(stack=0, head=0),
}

REFILL_BAD = {
    "src_slot -1": dict(src_slot=-1),
    "src_slot == stack": dict(src_slot=S),
    "src_slot past a stack of 1": dict(src_slot=1, stack=1),
    "padded_dim 200": dict(padded_dim=200),
    "padded_dim 0": dict(padded_dim=0),
    "ring + 8": dict(ring=RING + 8),
    "NULL ring": dict(ring=None),
    "num 0": dict(num=0),
}


@pytest.mark.parametrize("case", list(GATHER_BAD))
def test_ring_gather_rejects_bad_arguments_without_a_launch(case):
    from hanabizero_b200 import _lib
    lib = _lib.load()
    before = lib.hz_launch_count()
    assert _gather(**GATHER_BAD[case]) == _lib.HZ_ERR_ARG
    assert b"hz_ring_gather" in lib.hz_last_error()
    assert lib.hz_launch_count() == before


@pytest.mark.parametrize("case", list(REFILL_BAD))
def test_ring_refill_rejects_bad_arguments_without_a_launch(case):
    from hanabizero_b200 import _lib
    lib = _lib.load()
    before = lib.hz_launch_count()
    assert _refill(**REFILL_BAD[case]) == _lib.HZ_ERR_ARG
    assert b"hz_ring_refill" in lib.hz_last_error()
    assert lib.hz_launch_count() == before
