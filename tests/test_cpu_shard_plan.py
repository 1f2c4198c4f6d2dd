"""CPU: the host side of the sharded decode -- the range cutter, the scatter of an assembled body over gloo,
the tail-fetch plan (which rank sends which payload bytes to whom) and the output placement, for worlds 2-4,
empty ranks, and a copied-through package whose payload runs over several ranks."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from adaptive_compression_b200 import _lib as L
from adaptive_compression_b200 import distributed as D

MB = 4
HDR = MB + 14


@pytest.mark.parametrize("world", [2, 3, 4])
def test_body_ranges_cover_the_body(world):
    for n in (0, 1, world - 1, world, 100, 12345, (1 << 32) + 7):
        rs = D.body_ranges(n, world)
        assert len(rs) == world and rs[0][0] == 0 and rs[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(rs, rs[1:]))
        sizes = [hi - lo for lo, hi in rs]
        assert max(sizes) - min(sizes) <= 1
        for lo, hi in rs:
            b0, b1 = D.buffer_span(lo, hi, n, MB)
            assert b0 == lo and b1 == min(hi + MB + 13, n)


def test_tail_fetch_plan_exact_cover():
    rs = np.random.RandomState(1)
    for _ in range(300):
        world = int(rs.randint(2, 5))
        n = int(rs.randint(0, 3000))
        cuts = [0] + sorted(int(x) for x in rs.randint(0, n + 1, world - 1)) + [n]  # empty ranks included
        ranges = list(zip(cuts[:-1], cuts[1:]))
        needs = []
        for lo, hi in ranges:
            f0 = D.buffer_span(lo, hi, n, MB)[1]
            needs.append(int(rs.randint(0, n - f0 + 1)) if n > f0 and rs.rand() < 0.6 else 0)
        plan = D.tail_fetch_plan(ranges, needs, n, MB)
        got = {r: [] for r in range(world)}
        for src, dst, g0, g1 in plan:
            assert src > dst and g1 > g0
            assert ranges[src][0] <= g0 and g1 <= ranges[src][1]  # a sender only sends bytes of its own range
            got[dst].append((g0, g1))
        for r, ((lo, hi), need) in enumerate(zip(ranges, needs)):
            segs = sorted(got[r])
            f0 = D.buffer_span(lo, hi, n, MB)[1]
            pos = f0
            for g0, g1 in segs:
                assert g0 == pos
                pos = g1
            assert pos == f0 + need


def test_tail_fetch_plan_from_several_ranks():
    ranges = [(0, 100), (100, 100), (100, 150), (150, 400)]
    # rank 0 holds [0, 117) with the halo; its package needs body bytes up to 300
    plan = D.tail_fetch_plan(ranges, [183, 0, 0, 0], 400, MB)
    assert plan == [(2, 0, 117, 150), (3, 0, 150, 300)]


def _state(next_pos=0, out_before=0, pkg=None, status=L.RANGE_RUNNING):
    s = L.RangeState(next_pos, out_before, L.RANGE_NO_PKG, 0, 0, 0, 0, status)
    if pkg:
        s.pkg_pos, s.pkg_out, s.pkg_type, s.pkg_orig, s.pkg_comp = pkg
    return s


def test_output_placement_raw_package_over_several_ranks():
    # packages: [0, 22) a 4-byte native package (output [0, 4)); [22, 22 + 18 + 300000) a raw package
    # (output [4, 300004)); then a native package of 4 output bytes and END.
    raw_hdr, comp = 22, 300000
    pay = raw_hdr + HDR
    after = pay + comp
    body_len = after + 22 + 16
    orig = 4 + comp + 4
    ranges = [(0, 1000), (1000, 1000), (1000, 150000), (150000, 290000), (290000, body_len)]
    carried = (raw_hdr, 4, 255, comp, comp)
    entries = [_state(), _state(pay + comp, 4 + comp, carried), _state(pay + comp, 4 + comp, carried),
               _state(pay + comp, 4 + comp, carried), _state(pay + comp, 4 + comp, carried)]
    sl = D.output_slices(entries, ranges, orig, MB)
    assert sl == [(0, 4 + 1000 - pay), (4 + 1000 - pay, 4 + 1000 - pay), (4 + 1000 - pay, 4 + 150000 - pay),
                  (4 + 150000 - pay, 4 + 290000 - pay), (4 + 290000 - pay, orig)]
    # copied through because the type is unknown: the same placement with the payload length as output
    entries_u = [_state()] + [_state(pay + comp, 4 + comp, (raw_hdr, 4, 9, 77, comp))] * 4
    assert D.output_slices(entries_u, ranges, orig, MB) == sl
    # a decoded package (type 1) spanning ranks: its output belongs to the rank holding its header
    entries_d = [_state()] + [_state(pay + comp, 4 + 8192, (raw_hdr, 4, 1, 8192, comp))] * 4
    assert D.output_slices(entries_d, ranges, 4 + 8192 + 4, MB) == [(0, 8196), (8196, 8196), (8196, 8196), (8196, 8196),
                                                                   (8196, 8200)]
    # the walk ended inside rank 0 (END): every later slice is empty and the last rank owns the zero tail
    done = _state(40, 4, None, L.RANGE_END)
    assert D.output_slices([_state(), done, done, done, done], ranges, 100, MB) == [(0, 4), (4, 4), (4, 4), (4, 4), (4, 100)]
    # a raw package cut by orig_size inside rank 0's bytes: every later slice is empty
    short = 4 + 500
    assert D.output_slices(entries, ranges, short, MB) == [(0, short)] + [(short, short)] * 4
    # cut inside rank 2's bytes
    cut = 4 + 100000
    assert D.output_slices(entries, ranges, cut, MB) == [sl[0], sl[1], (sl[2][0], cut), (cut, cut), (cut, cut)]


def test_state_words_round_trip():
    s = _state(123, 456, (7, 8, 255, 9, 10), L.RANGE_COMPLETE)
    t = D.state_from_words(D.state_to_words(s))
    assert bytes(s) == bytes(t)
    u = _state()
    w = D.state_to_words(u)
    assert w[2] == -1 and bytes(D.state_from_words(w)) == bytes(u)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, body, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        t = torch.from_numpy(np.frombuffer(body, dtype=np.uint8).copy()) if rank == 0 else None
        buf = D.scatter_body(t, len(body), src=0, marker_bytes=MB)
        q.put((rank, buf.numpy().tobytes()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n", [(2, 1000), (3, 5), (4, 40), (4, 3001)])
def test_scatter_body_over_gloo(world, n):
    body = bytes(np.random.RandomState(n).randint(0, 256, n, dtype=np.uint8))
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, body, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for r, (lo, hi) in enumerate(D.body_ranges(n, world)):
        b0, b1 = D.buffer_span(lo, hi, n, MB)
        assert res[r] == body[b0:b1]
