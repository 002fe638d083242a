"""CPU: the parts of the reanalyze pipeline that need no device — the ctypes mirror of hz_policy_ticket, the argument
checks of hz_obs_pack_windows and hz_wave_policy (nothing launched), and SearchPipeline.submit_observations /
ReanalyzePipeline.submit rejecting bad windows, legal moves, masks and policy outputs before a ticket takes a wave
position."""
import ctypes
import os
import subprocess

import pytest
import torch

from helpers import ROOT


def test_policy_ticket_mirrors_the_header_layout(tmp_path):
    from hanabizero_b200 import _lib
    cls = _lib.PolicyTicket
    lines = ['printf("%zu", sizeof(hz_policy_ticket));']
    lines += [f'printf(" %zu", offsetof(hz_policy_ticket, {f}));' for f, _ in cls._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hzb200.h"\nint main(void) {\n' + "\n".join(lines)
                   + "\nreturn 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert ctypes.sizeof(cls) == out[0] == 16
    assert [getattr(cls, f).offset for f, _ in cls._fields_] == out[1:] == [0, 8]
    assert 64 * ctypes.sizeof(cls) == 1024       # the table travels in the kernel parameters


def _layout(**over):
    from hanabizero_b200 import _lib
    f = dict(stack=4, frame_dim=785, frame_stride=800, elem_bytes=2, frame_words=25, bit_offset=0)
    f.update(over)
    return _lib.ObsLayout(**f)


def _ticket(**over):
    """A window of 4 + 6 - 1 = 9 Hanabi-Full frames per row."""
    from hanabizero_b200 import _lib
    f = dict(obs=0x1000, ld_obs=9 * 785, legal=0x2000, ld_legal=20, noise=None, obs_format=_lib.HZ_OBS_F32,
             legal_format=_lib.HZ_LEGAL_I32)
    f.update(over)
    return _lib.ObsTicket(**f)


def test_obs_pack_windows_rejects_bad_arguments_before_touching_a_device():
    from hanabizero_b200 import _lib
    lib = _lib.load()
    before = lib.hz_launch_count()
    buf = ctypes.c_void_p(0x1000)

    def pack(tickets=None, count=1, slots=2, n=60, a=20, layout=None, positions=6, x=buf, legal=buf, table=True):
        tab = (_lib.ObsTicket * max(1, len(tickets or [0])))(*(tickets or [_ticket()])) if table else None
        lay = ctypes.byref(layout if layout is not None else _layout())
        return lib.hz_obs_pack_windows(None, 0, tab, count, slots, n, a, lay, positions, x, legal, buf)

    F32, U8, BITS = _lib.HZ_OBS_F32, _lib.HZ_OBS_U8, _lib.HZ_OBS_BITS
    cases = [
        (dict(table=False), b"NULL ticket table"),
        (dict(count=3), b"count"), (dict(count=0), b"count"), (dict(slots=65), b"slots"),
        (dict(n=0), b"n = 0"), (dict(slots=64, n=1 << 19), b"slots * n"),
        (dict(n=62), b"not a multiple of positions"), (dict(n=6, positions=4), b"not a multiple of positions"),
        (dict(positions=0), b"positions"), (dict(positions=-6), b"positions"), (dict(n=6, positions=12), b"positions"),
        (dict(a=33), b"num_actions"), (dict(a=0), b"num_actions"),
        (dict(layout=_layout(stack=0)), b"stack"), (dict(layout=_layout(frame_stride=808)), b"frame_stride"),
        (dict(layout=_layout(frame_dim=801)), b"frame_dim"), (dict(layout=_layout(elem_bytes=1)), b"elem_bytes"),
        (dict(x=None), b"NULL staging"), (dict(legal=None), b"NULL staging"),
        (dict(tickets=[_ticket(obs=None)]), b"ticket 0 has a NULL input"),
        (dict(tickets=[_ticket(), _ticket(legal=None)], count=2), b"ticket 1 has a NULL input"),
        (dict(tickets=[_ticket(obs_format=3)]), b"obs_format"), (dict(tickets=[_ticket(obs_format=-1)]), b"obs_format"),
        (dict(tickets=[_ticket(legal_format=3)]), b"legal_format"),
        (dict(tickets=[_ticket(legal_format=-1)]), b"legal_format"),
        # ld_obs shorter than the window (long enough for a stack of 4) in every format
        (dict(tickets=[_ticket(ld_obs=9 * 785 - 1)]), b"elements of a window"),
        (dict(tickets=[_ticket(ld_obs=4 * 785)]), b"elements of a window"),
        (dict(tickets=[_ticket(obs_format=U8, ld_obs=9 * 785 - 1)]), b"elements of a window"),
        (dict(tickets=[_ticket(obs_format=BITS, ld_obs=9 * 25 - 1)]), b"elements of a window"),
        (dict(tickets=[_ticket(obs_format=BITS, ld_obs=4 * 25)]), b"elements of a window"),
        (dict(tickets=[_ticket(ld_obs=5 * 785)], positions=3), b"elements of a window"),
        (dict(tickets=[_ticket(ld_legal=19)]), b"ld_legal"),
        (dict(tickets=[_ticket(obs_format=BITS, ld_obs=225)], layout=_layout(frame_words=0)), b"frame_words"),
        (dict(tickets=[_ticket(obs_format=BITS, ld_obs=225)], layout=_layout(bit_offset=-1)), b"bit_offset"),
    ]
    for kw, msg in cases:
        assert pack(**kw) == _lib.HZ_ERR_ARG, kw
        assert msg in lib.hz_last_error(), (kw, lib.hz_last_error())
    assert lib.hz_obs_pack_windows(None, 0, (_lib.ObsTicket * 1)(_ticket()), 1, 1, 60, 20, None, 6, buf, buf,
                                   buf) == _lib.HZ_ERR_ARG
    assert b"NULL layout" in lib.hz_last_error()
    assert lib.hz_launch_count() == before


def test_wave_policy_rejects_bad_arguments_before_touching_a_device():
    from hanabizero_b200 import _lib
    lib = _lib.load()
    before = lib.hz_launch_count()
    good = _lib.PolicyTicket(mask=0x3000, out=0x4000)

    def policy(tickets=None, count=1, slots=2, n=64, a=20, stats=0x1000, table=True):
        tickets = tickets or [good]
        tab = (_lib.PolicyTicket * len(tickets))(*tickets) if table else None
        return lib.hz_wave_policy(None, 0, tab, count, slots, n, a, stats)

    cases = [
        (dict(table=False), b"NULL ticket table"),
        (dict(count=3), b"count"), (dict(count=0), b"count"), (dict(slots=0), b"slots"), (dict(slots=65), b"slots"),
        (dict(n=0), b"n = 0"), (dict(slots=64, n=1 << 19), b"slots * n"),
        (dict(a=0), b"num_actions"), (dict(a=33), b"num_actions"),
        (dict(stats=None), b"NULL statistics"),
        (dict(tickets=[_lib.PolicyTicket(mask=0x3000, out=None)]), b"ticket 0 has a NULL output"),
        (dict(tickets=[good, _lib.PolicyTicket(mask=None, out=None)], count=2), b"ticket 1 has a NULL output"),
    ]
    for kw, msg in cases:
        assert policy(**kw) == _lib.HZ_ERR_ARG, kw
        assert msg in lib.hz_last_error(), (kw, lib.hz_last_error())
    assert lib.hz_launch_count() == before


class _Plan:
    frame_stride = 800


def _pipeline(n=24, stack=4):
    """A SearchPipeline with only what submit_observations reads before a ticket takes a position (no device)."""
    from hanabizero_b200.mcts import SearchPipeline, WaveSchedule
    p = SearchPipeline.__new__(SearchPipeline)
    p.n, p.a, p.wave, p.depth, p.stack = n, 20, 4, 2, stack
    p.frame_dim, p.frame_words = 785, 25
    p._iplan = _Plan()
    p.device = torch.device("cuda", 0)
    p._waves = WaveSchedule(p.wave, p.depth)
    p.submitted = 0
    return p


def test_submit_observations_rejects_bad_windows_and_policy_arguments():
    n, a, S, D, W, P = 24, 20, 4, 785, 25, 6
    p = _pipeline()
    good = dict(fraction=0.25, noises=None, obs=torch.zeros(n // P, S + P - 1, D), legal=torch.zeros(n, a),
                positions=P, out_policy=torch.zeros(n, a, dtype=torch.float64), policy_mask=torch.ones(n, dtype=torch.uint8))
    bad = [
        dict(positions=0), dict(positions=5), dict(positions=48),
        dict(obs=torch.zeros(n // P, S + P, D)), dict(obs=torch.zeros(n // P, S + P - 2, D)),
        dict(obs=torch.zeros(n // P + 1, S + P - 1, D)), dict(obs=torch.zeros(n, S, D)),       # stacks, not windows
        dict(obs=torch.zeros(n // P, (S + P - 1) * D + 1)),
        dict(obs=torch.zeros(n // P, S + P - 1, D, dtype=torch.uint8)[:, :, :D - 1]),
        dict(obs=torch.zeros(n // P, S + P - 1, D, dtype=torch.int32)),                        # bits are [.., W]
        dict(obs=torch.zeros(n // P, (S + P - 1) * W - 1, dtype=torch.int32)),
        dict(obs=torch.zeros(n // P, S + P - 1, D), positions=3),
        dict(legal=torch.zeros(n // P, a)), dict(legal=torch.zeros(n, a + 1)), dict(legal=torch.zeros(n // P, P, a)),
        dict(legal=torch.zeros(n)),
        dict(out_policy=torch.zeros(n, a + 1, dtype=torch.float64)), dict(out_policy=torch.zeros(n, a)),
        dict(out_policy=torch.zeros(n, a, dtype=torch.float64).numpy()),
        dict(policy_mask=torch.ones(n + 1, dtype=torch.uint8)), dict(policy_mask=torch.ones(n // P, dtype=torch.uint8)),
        dict(out_policy=None),                                                                 # a mask without targets
    ]
    for kw in bad:
        args = dict(good)
        args.update(kw)
        with pytest.raises(ValueError):
            p.submit_observations(**args)
        assert p._waves.open is None and p.submitted == 0, kw


class _Config:
    action_space_size = 20
    root_exploration_fraction = 0.25
    root_dirichlet_alpha = 0.3


def test_reanalyze_submit_rejects_bad_shapes_before_taking_a_ticket():
    from hanabizero_b200.reanalyze import ReanalyzePipeline
    batch, K, S, D, A = 4, 5, 4, 785, 20
    rp = ReanalyzePipeline.__new__(ReanalyzePipeline)
    rp.config, rp.batch, rp.per, rp.stack, rp.a = _Config(), batch, K + 1, S, A
    rp.roots = batch * (K + 1)
    rp.pipe = _pipeline(n=rp.roots, stack=S)
    rp.device, rp._out = rp.pipe.device, {}
    good = dict(obs_windows=torch.zeros(batch, K + S, D, dtype=torch.uint8), legal_actions=torch.zeros(batch, K + 1, A),
                policy_mask=torch.ones(batch, K + 1))
    bad = [
        dict(obs_windows=torch.zeros(batch, K + S + 1, D, dtype=torch.uint8)),
        dict(obs_windows=torch.zeros(batch, S, D, dtype=torch.uint8)),
        dict(obs_windows=torch.zeros(batch + 1, K + S, D, dtype=torch.uint8)),
        dict(obs_windows=torch.zeros(batch * (K + 1), S, D)),                     # expanded stacks
        dict(obs_windows=torch.zeros(batch, (K + S) * 25 + 1, dtype=torch.int32)),
        dict(legal_actions=torch.zeros(batch, K, A)), dict(legal_actions=torch.zeros(batch, K + 1, A + 1)),
        dict(legal_actions=torch.zeros(batch * (K + 1), A)), dict(legal_actions=torch.zeros(batch, K + 1)),  # float words
        dict(legal_actions=torch.zeros(batch, K + 2, dtype=torch.int32)),
        dict(policy_mask=torch.ones(batch, K)), dict(policy_mask=torch.ones(batch * (K + 1))),
    ]
    for kw in bad:
        args = dict(good)
        args.update(kw)
        with pytest.raises(ValueError):
            rp.submit(**args)
        assert rp.pipe._waves.open is None and rp.pipe.submitted == 0 and not rp._out, kw
