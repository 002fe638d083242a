"""CPU: the parts of observation tickets that need no device — the ctypes mirrors of hz_obs_ticket / hz_obs_layout, the
argument checks of hz_obs_pack, and SearchPipeline.submit_observations rejecting bad arguments before the ticket takes
a wave position."""
import ctypes
import os
import subprocess

import pytest
import torch

from helpers import ROOT


@pytest.mark.parametrize("name,cls_name,size", [("hz_obs_ticket", "ObsTicket", 48), ("hz_obs_layout", "ObsLayout", 24)])
def test_obs_structs_mirror_the_header_layout(tmp_path, name, cls_name, size):
    from hanabizero_b200 import _lib
    cls = getattr(_lib, cls_name)
    lines = [f'printf("%zu", sizeof({name}));']
    lines += [f'printf(" %zu", offsetof({name}, {f}));' for f, _ in cls._fields_]
    lines += ['printf(" %d %d %d %d %d %d", HZ_OBS_F32, HZ_OBS_U8, HZ_OBS_BITS, HZ_LEGAL_I32, HZ_LEGAL_F32, HZ_LEGAL_MASK);']
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hzb200.h"\nint main(void) {\n' + "\n".join(lines)
                   + "\nreturn 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    k = len(cls._fields_)
    assert ctypes.sizeof(cls) == int(out[0]) == size
    assert [getattr(cls, f).offset for f, _ in cls._fields_] == [int(o) for o in out[1:1 + k]]
    assert [int(c) for c in out[1 + k:]] == [_lib.HZ_OBS_F32, _lib.HZ_OBS_U8, _lib.HZ_OBS_BITS, _lib.HZ_LEGAL_I32,
                                             _lib.HZ_LEGAL_F32, _lib.HZ_LEGAL_MASK]
    # 64 tickets and the other kernel parameters fit the 4 KB the header promises
    assert 64 * ctypes.sizeof(_lib.ObsTicket) <= 4096


def _layout(**over):
    from hanabizero_b200 import _lib
    f = dict(stack=4, frame_dim=785, frame_stride=800, elem_bytes=2, frame_words=25, bit_offset=0)
    f.update(over)
    return _lib.ObsLayout(**f)


def _ticket(**over):
    from hanabizero_b200 import _lib
    f = dict(obs=0x1000, ld_obs=4 * 785, legal=0x2000, ld_legal=20, noise=None, obs_format=_lib.HZ_OBS_F32,
             legal_format=_lib.HZ_LEGAL_I32)
    f.update(over)
    return _lib.ObsTicket(**f)


def test_obs_pack_rejects_bad_arguments_before_touching_a_device():
    from hanabizero_b200 import _lib
    lib = _lib.load()
    before = lib.hz_launch_count()
    buf = ctypes.c_void_p(0x1000)

    def pack(tickets=None, count=1, slots=2, n=64, a=20, layout=None, x=buf, legal=buf, table=True):
        tab = (_lib.ObsTicket * max(1, len(tickets or [0])))(*(tickets or [_ticket()])) if table else None
        lay = ctypes.byref(layout if layout is not None else _layout())
        return lib.hz_obs_pack(None, 0, tab, count, slots, n, a, lay, x, legal, buf)

    F32, U8, BITS = _lib.HZ_OBS_F32, _lib.HZ_OBS_U8, _lib.HZ_OBS_BITS
    cases = [
        (dict(table=False), b"NULL ticket table"),
        (dict(count=3), b"count"), (dict(count=0), b"count"), (dict(slots=65), b"slots"),
        (dict(n=0), b"n = 0"), (dict(slots=64, n=1 << 19), b"slots * n"),
        (dict(a=33), b"num_actions"), (dict(a=0), b"num_actions"),
        (dict(layout=_layout(stack=0)), b"stack"), (dict(layout=_layout(stack=65)), b"stack"),
        (dict(layout=_layout(frame_stride=808)), b"frame_stride"),
        (dict(layout=_layout(frame_stride=0)), b"frame_stride"),
        (dict(layout=_layout(stack=64, frame_stride=1040)), b"frame_stride"),
        (dict(layout=_layout(frame_dim=801)), b"frame_dim"), (dict(layout=_layout(frame_dim=0)), b"frame_dim"),
        (dict(layout=_layout(elem_bytes=1)), b"elem_bytes"),
        (dict(x=None), b"NULL staging"), (dict(legal=None), b"NULL staging"),
        (dict(tickets=[_ticket(obs=None)]), b"ticket 0 has a NULL input"),
        (dict(tickets=[_ticket(), _ticket(legal=None)], count=2), b"ticket 1 has a NULL input"),
        (dict(tickets=[_ticket(obs_format=3)]), b"obs_format"),
        (dict(tickets=[_ticket(obs_format=-1)]), b"obs_format"),
        (dict(tickets=[_ticket(legal_format=3)]), b"legal_format"),
        (dict(tickets=[_ticket(ld_obs=4 * 785 - 1)]), b"ld_obs"),
        (dict(tickets=[_ticket(obs_format=U8, ld_obs=4 * 785 - 1)]), b"ld_obs"),
        (dict(tickets=[_ticket(obs_format=BITS, ld_obs=99)]), b"ld_obs"),
        (dict(tickets=[_ticket(ld_legal=19)]), b"ld_legal"),
        (dict(tickets=[_ticket(legal_format=_lib.HZ_LEGAL_MASK, ld_legal=0)]), b"ld_legal"),
        # bit frames: the frame must lie inside the packed string (Hanabi-Full local: 660 bits from 125 in 25 words)
        (dict(tickets=[_ticket(obs_format=BITS, ld_obs=100)], layout=_layout(frame_words=0)), b"frame_words"),
        (dict(tickets=[_ticket(obs_format=BITS, ld_obs=100)], layout=_layout(bit_offset=-1)), b"bit_offset"),
        (dict(tickets=[_ticket(obs_format=BITS, ld_obs=100)], layout=_layout(frame_dim=660, frame_stride=672,
                                                                              bit_offset=141)), b"bit_offset"),
        (dict(tickets=[_ticket(obs_format=BITS, ld_obs=100)], layout=_layout(frame_words=24)), b"bit_offset"),
    ]
    for kw, msg in cases:
        assert pack(**kw) == _lib.HZ_ERR_ARG, kw
        assert msg in lib.hz_last_error(), (kw, lib.hz_last_error())
    assert lib.hz_obs_pack(None, 0, (_lib.ObsTicket * 1)(_ticket()), 1, 1, 64, 20, None, buf, buf, buf) == _lib.HZ_ERR_ARG
    assert b"NULL layout" in lib.hz_last_error()
    assert lib.hz_launch_count() == before


class _Plan:
    frame_stride = 800


def _pipeline(stack=4):
    """A SearchPipeline with only what submit_observations reads before a ticket takes a position (no device)."""
    from hanabizero_b200.mcts import SearchPipeline, WaveSchedule
    p = SearchPipeline.__new__(SearchPipeline)
    p.n, p.a, p.wave, p.depth, p.stack = 8, 20, 4, 2, stack
    p.frame_dim, p.frame_words = 785, 25
    p._iplan = None if stack is None else _Plan()
    p.device = torch.device("cuda", 0)
    p._waves = WaveSchedule(p.wave, p.depth)
    p.submitted = 0
    return p


def test_submit_observations_rejects_bad_arguments_before_taking_a_ticket():
    n, a, S, D, W = 8, 20, 4, 785, 25
    with pytest.raises(RuntimeError, match="stack="):
        _pipeline(stack=None).submit_observations(0.25, None, torch.zeros(n, S, D), torch.zeros(n, a))
    p = _pipeline()
    good_obs, good_legal = torch.zeros(n, S, D), torch.zeros(n, a, dtype=torch.int32)
    bad = [
        dict(obs=torch.zeros(n, S, D + 1)), dict(obs=torch.zeros(n + 1, S * D)), dict(obs=torch.zeros(n, S - 1, D)),
        dict(obs=torch.zeros(n, S, D, dtype=torch.uint8)[:, :, :D - 1]),
        dict(obs=torch.zeros(n, S, D, dtype=torch.int32)),                    # int32 frames are packed bits: [n, S, W]
        dict(obs=torch.zeros(n, S * W + 1, dtype=torch.int32)),
        dict(legal=torch.zeros(n, a + 1)), dict(legal=torch.zeros(n + 1, dtype=torch.int32)),
        dict(legal=torch.zeros(n)),                                           # a bit mask is int32
        dict(legal=torch.zeros(n, 2, a)),
        dict(noises=torch.zeros(n, a - 1)),
        dict(out_visits=torch.zeros(n, a + 1, dtype=torch.int32)), dict(out_values=torch.zeros(n + 1)),
    ]
    for kw in bad:
        args = dict(fraction=0.25, noises=None, obs=good_obs, legal=good_legal)
        args.update(kw)
        with pytest.raises(ValueError):
            p.submit_observations(**args)
        assert p._waves.open is None and p.submitted == 0, kw
