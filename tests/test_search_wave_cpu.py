"""CPU: the parts of search waves that need no device — argument checks of hz_wave_pack / hz_wave_unpack, the ctypes
mirror of hz_wave_ticket, the ticket-id and wave-closing rules of SearchPipeline(wave=G), and the carving of one
ticket's rows out of a gathered wave under gloo with world size 2."""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import ROOT


def test_wave_calls_reject_bad_sizes_before_touching_a_device():
    from hanabizero_b200 import _lib
    lib = _lib.load()
    before = lib.hz_launch_count()
    table = (_lib.WaveTicket * 2)()
    buf = ctypes.c_void_p(0x1000)
    pack = lambda tab, count, slots, n, a, hrb: lib.hz_wave_pack(None, 0, tab, count, slots, n, a, hrb, buf, buf, buf,
                                                                 buf, buf)
    cases = [((None, 1, 1, 64, 20, 1024), b"NULL ticket table"),
             ((table, 3, 2, 64, 20, 1024), b"count"),
             ((table, 0, 2, 64, 20, 1024), b"count"),
             ((table, 2, 65, 64, 20, 1024), b"slots"),
             ((table, 2, 2, 0, 20, 1024), b"n = 0"),
             ((table, 2, 64, 1 << 19, 20, 1024), b"slots * n"),
             ((table, 2, 2, 64, 33, 1024), b"num_actions"),
             ((table, 2, 2, 64, 0, 1024), b"num_actions"),
             ((table, 2, 2, 64, 20, 1000), b"hidden_row_bytes"),
             ((table, 2, 2, 64, 20, 1 << 17), b"hidden_row_bytes")]
    for args, msg in cases:
        assert pack(*args) == _lib.HZ_ERR_ARG, args
        assert msg in lib.hz_last_error(), (args, lib.hz_last_error())
    assert lib.hz_wave_pack(None, 0, table, 1, 2, 64, 20, 1024, buf, None, buf, buf, buf) == _lib.HZ_ERR_ARG
    assert b"NULL staging" in lib.hz_last_error()
    assert pack(table, 1, 2, 64, 20, 1024) == _lib.HZ_ERR_ARG           # ticket 0 has no inputs
    assert b"ticket 0" in lib.hz_last_error()
    assert lib.hz_wave_unpack(None, 0, None, 1, 1, 64, 20, buf) == _lib.HZ_ERR_ARG
    assert lib.hz_wave_unpack(None, 0, table, 2, 1, 64, 20, buf) == _lib.HZ_ERR_ARG
    assert lib.hz_wave_unpack(None, 0, table, 1, 1, 64, 20, None) == _lib.HZ_ERR_ARG
    assert b"statistics" in lib.hz_last_error()
    assert lib.hz_launch_count() == before


def test_wave_ticket_mirrors_the_header_layout(tmp_path):
    import subprocess
    from hanabizero_b200 import _lib
    cls = _lib.WaveTicket
    lines = ['printf("%zu", sizeof(hz_wave_ticket));']
    lines += [f'printf(" %zu", offsetof(hz_wave_ticket, {f}));' for f, _ in cls._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hzb200.h"\nint main(void) {\n' + "\n".join(lines)
                   + "\nreturn 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    size, *offsets = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert ctypes.sizeof(cls) == int(size) == 56
    assert [getattr(cls, f).offset for f, _ in cls._fields_] == [int(o) for o in offsets]


def test_wave_schedule_ticket_ids_and_closing_rules():
    from hanabizero_b200.mcts import WaveSchedule
    ws = WaveSchedule(wave=4, depth=3)
    ids = []
    for k in range(9):                                   # full waves: slots round robin, id = slot * G + position
        slot, p = ws.take(True, 0.25)
        ids.append(slot * ws.wave + p)
        if ws.full():
            assert ws.close()["count"] == 4
    assert ids == [0, 1, 2, 3, 4, 5, 6, 7, 8] and ws.is_open(2) and ws.slot_of(8) == 2
    assert not ws.closes(True, 0.25)
    assert ws.closes(False, 0.0) and ws.closes(True, 0.5)   # noise-ness or fraction differs: launch the open wave
    assert ws.close() == dict(slot=2, noisy=True, fraction=0.25, count=1)
    assert ws.open is None and not ws.closes(False, 0.0) and not ws.full()
    assert ws.take(False, 0.0) == (0, 0)                  # the next wave opens on the next slot
    assert not ws.is_open(2) and ws.slot_of(3) == 0
    one = WaveSchedule(wave=1, depth=3)                  # G = 1: the ticket is the slot index
    got = []
    for _ in range(4):
        got.append(one.take(True, 0.25))
        assert one.full()
        one.close()
    assert got == [(0, 0), (1, 0), (2, 0), (0, 0)]


def _worker(rank, world, port, G, n, A, out_q):
    from hanabizero_b200.dist import AsyncStatsGather, wave_rows
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(0)
    visits_all = rng.integers(0, 50, (world, G, n, A)).astype(np.int32)    # [rank][ticket] rows
    values_all = rng.standard_normal((world, G, n)).astype(np.float32)
    flat = torch.cat((torch.from_numpy(visits_all[rank]).reshape(-1),
                      torch.from_numpy(values_all[rank].view(np.int32).copy()).reshape(-1)))
    ag = AsyncStatsGather(G * n, A, torch.device("cpu"), depth=2)
    visits, values = ag.result(ag.submit_flat(flat))
    ok = True
    for p in range(G):
        v, val = wave_rows(visits, values, world, G, p)
        ok = ok and v.shape == (world * n, A) and val.shape == (world * n,)
        ok = ok and bool((v.numpy() == visits_all[:, p].reshape(world * n, A)).all())
        ok = ok and bool((val.numpy().view(np.uint32) == values_all[:, p].reshape(-1).view(np.uint32)).all())
    out_q.put((rank, ok))
    dist.barrier()
    dist.destroy_process_group()


def test_wave_rows_carves_a_ticket_out_of_the_gathered_wave_world2_gloo():
    world, G, n, A = 2, 3, 5, 20
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, world, port, G, n, A, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(ok for _, ok in res), res
