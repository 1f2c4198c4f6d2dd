"""GPU parity of the fixed-grid compress at file scale: bodies and counters of ambc_compress_dev and
ambc_compress_host against the oracle past one scan tile (2048 chunks), on the edges of the host path's upload
pieces, and past 1024 scan tiles, where k_scan_tiles carries its sum into a second pass.

Every chunk is encoded on its own, so one per-chunk-raw oracle run over a clean input gives every package; a chunk
overwritten with random bytes is run through the oracle alone.  In strict mode the body is then the packages before
the first chunk without a winner, one raw package for the rest of the file, and END."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle as O
import synth_ref

pytestmark = pytest.mark.gpu

MB = O.FIXED_MARKER
OVH = len(MB) + 14
END = MB + bytes(12)
TILE = 2048  # SCAN_TILE: chunks per scan tile


@pytest.fixture(scope="module")
def eng():
    from adaptive_compression_b200 import engine
    engine.require_cuda()
    return engine


def _oracle_slice(a, chunk):
    """orc_compress_body in per-chunk-raw mode on one chunk-aligned slice -> (body without END, types, comps)"""
    n = a.size
    cands = np.array([chunk], dtype=np.int64)
    meth = np.array(O.NATIVE, dtype=np.int32)
    mk = np.frombuffer(MB, dtype=np.uint8)
    cap = n // chunk + 4
    out = np.empty(n + cap * OVH + 64, dtype=np.uint8)
    mt, mo, mc = np.zeros(cap, np.int32), np.zeros(cap, np.int64), np.zeros(cap, np.int64)
    npk = O.C.c_long(0)
    r = O.lib().orc_compress_body(a.ctypes.data, n, cands.ctypes.data, 1, meth.ctypes.data, meth.size, mk.ctypes.data,
                                  mk.size, 1, out.ctypes.data, mt.ctypes.data, mo.ctypes.data, mc.ctypes.data, cap,
                                  O.C.byref(npk))
    k = npk.value
    return out[:r - len(END)], mt[:k].copy(), mc[:k].copy()


class Grid:
    """the oracle's per-chunk packages of an input: types, comps, and the per-chunk-raw body (without END) with the
    offset of every package"""

    def __init__(self, data, chunk):
        self.data, self.chunk, self.n = data, chunk, data.size
        n_chunks = -(-self.n // chunk)
        step = max(1, -(-n_chunks // (8 * (os.cpu_count() or 1)))) * chunk
        O.set_lz_fast(True)  # the oracle's indexed match search: the same bytes as the reference's scan, faster
        try:
            with ThreadPoolExecutor(os.cpu_count() or 1) as ex:  # (ctypes calls release the GIL)
                parts = list(ex.map(lambda b0: _oracle_slice(data[b0:b0 + step], chunk), range(0, self.n, step)))
        finally:
            O.set_lz_fast(False)
        self.body = np.concatenate([p[0] for p in parts])
        self.types = np.concatenate([p[1] for p in parts])
        self.comps = np.concatenate([p[2] for p in parts])
        assert self.types.size == n_chunks
        self.offs = np.zeros(n_chunks + 1, dtype=np.int64)
        np.cumsum(self.comps + OVH, out=self.offs[1:])

    def copy(self, data):
        g = Grid.__new__(Grid)
        g.__dict__.update(self.__dict__, data=data, types=self.types.copy(), comps=self.comps.copy(), offs=self.offs.copy())
        return g

    def patch(self, chunks):
        """the grid of the input with `chunks` overwritten in place: their packages rerun through the oracle"""
        for i in sorted(chunks):
            b0 = i * self.chunk
            body, t, c = _oracle_slice(self.data[b0:b0 + self.chunk], self.chunk)
            o0, o1 = self.offs[i], self.offs[i + 1]
            self.body = np.concatenate([self.body[:o0], body, self.body[o1:]])
            self.types[i], self.comps[i] = t[0], c[0]
            self.offs[i + 1:] += (c[0] + OVH) - (o1 - o0)

    def expect(self, pcr):
        """-> (body bytes, first_raw, n_packages, usage, payload_bytes) the library must report"""
        raw = np.flatnonzero(self.types == 255)
        fr = int(raw[0]) if raw.size else -1
        last = self.types.size if (pcr or fr < 0) else fr
        t, c = self.types[:last], self.comps[:last]
        usage = [int((t == 255).sum())] + [int((t == m).sum()) for m in (1, 2, 3, 4)]
        payload = int(c[(t >= 1) & (t <= 4)].sum())
        body = self.body[:self.offs[last]].tobytes()
        if not pcr and fr >= 0:
            rest = self.n - fr * self.chunk
            body += MB + bytes([255, 0]) + rest.to_bytes(4, "little") * 3 + self.data[fr * self.chunk:].tobytes()
            usage[0] = 1
        return body + END, fr, last + (1 if not pcr and fr >= 0 else 0), usage, payload


def piece_starts(n, chunk):
    """the upload pieces of ambc_compress_host (api.cu), as chunk indices: whole scan tiles that ramp up from 8 MiB
    to 64 MiB and back down when the input is large enough, equal 64 MiB pieces otherwise"""
    n_tiles = -(-(-(-n // chunk)) // TILE)
    tile_bytes = TILE * chunk
    unit = max(1, (8 << 20) // tile_bytes)
    big = max(unit, (64 << 20) // tile_bytes)
    while True:
        ramp, r = [], unit
        while r < big:
            ramp.append(r)
            r *= 2
        if n_tiles >= 2 * sum(ramp) + big:
            mid = n_tiles - 2 * sum(ramp)
            sizes = list(ramp)
            while mid >= 2 * big:
                sizes.append(big)
                mid -= big
            sizes += [mid] + ramp[::-1]
        else:
            sizes = [min(big, n_tiles - t) for t in range(0, n_tiles, big)]
        if len(sizes) <= 64:
            break
        big *= 2
    return [int(x) * TILE for x in np.cumsum([0] + sizes)]


def _noise(data, chunk, chunks, seed):
    r = np.random.RandomState(seed)
    for i in chunks:
        seg = data[i * chunk:(i + 1) * chunk]
        seg[:] = r.randint(0, 256, size=seg.size).astype(np.uint8)


def _run_both(eng, data, chunk, pcr, want, label):
    from adaptive_compression_b200 import _lib as L
    body, fr, npk, usage, payload = want
    flags = L.F_PER_CHUNK_RAW if pcr else 0
    o = eng.compress_device(eng.to_device(data), chunk, flags=flags)
    got = o.body.cpu().numpy().tobytes()
    assert (got == body, o.first_raw, o.n_packages, list(o.usage), o.payload_bytes) == (True, fr, npk, usage, payload), \
        (label, "dev", len(got), len(body))
    del o
    hb, res, _, _ = eng.compress_host(data, data.size, chunk, flags=flags)
    got = hb.tobytes()
    assert (got == body, res.first_raw, res.n_packages, list(res.usage), res.payload_bytes) == \
        (True, fr, npk, usage, payload), (label, "host", len(got), len(body))


def _strict_first_raw_cases(eng, n, chunk, at, seed):
    """strict mode, first chunk without a winner at each of `at` in turn"""
    data = synth_ref.corpus(n, 0)
    grid = Grid(data, chunk)
    assert not (grid.types == 255).any()
    clean = data.copy()
    for k, i in enumerate(at):
        _noise(data, chunk, [i], seed + k)
        g = grid.copy(data)
        g.patch([i])
        want = g.expect(False)
        assert want[1] == i, (i, want[1])
        _run_both(eng, data, chunk, False, want, "first raw %d" % i)
        data[:] = clean
    return grid, data


def test_strict_first_raw_on_tile_and_piece_edges_equal_pieces(eng):
    """just over 64 MiB of 4 KiB chunks: two upload pieces (64 MiB, then the rest) and a short last chunk"""
    chunk = 4096
    n = (64 << 20) + 5 * chunk + 1000
    starts = piece_starts(n, chunk)
    n_chunks = -(-n // chunk)
    assert starts[:2] == [0, 16384] and len(starts) == 3 and starts[-1] >= n_chunks
    at = [0, 1, TILE - 1, TILE, TILE + 1, starts[1] - 1, starts[1], n_chunks - 1]
    grid, data = _strict_first_raw_cases(eng, n, chunk, at, 700)
    # per-chunk-raw mode: raw chunks on both sides of tile and piece edges in one file
    raw = [TILE - 1, TILE, 2 * TILE - 1, 2 * TILE, starts[1] - 1, starts[1], n_chunks - 1]
    _noise(data, chunk, raw, 710)
    grid.data = data
    grid.patch(raw)
    want = grid.expect(True)
    assert want[1] == TILE - 1 and want[3][0] == len(raw)
    _run_both(eng, data, chunk, True, want, "pcr tile edges")


def test_strict_first_raw_on_piece_edges_ramp_plan(eng):
    """176 MiB of 4 KiB chunks: the ramp plan, pieces of 1, 2, 4, 8, 4, 2 and 1 tiles"""
    chunk = 4096
    n = 176 << 20
    starts = piece_starts(n, chunk)
    assert [b - a for a, b in zip(starts, starts[1:])] == [TILE * k for k in (1, 2, 4, 8, 4, 2, 1)]
    n_chunks = n // chunk
    _strict_first_raw_cases(eng, n, chunk, [starts[3], starts[4] - 1, starts[6], n_chunks - 1], 720)


def test_per_chunk_raw_past_1024_scan_tiles(eng):
    """chunk 64, per-chunk-raw mode, 1029 scan tiles plus a short chunk: k_scan_tiles of the device path makes a
    second pass over the tile sums with the carry of the first"""
    chunk = 64
    n = (1024 + 5) * TILE * chunk + 37
    n_chunks = -(-n // chunk)
    assert -(-n_chunks // TILE) > 1024
    data = synth_ref.corpus(n, 0)
    grid = Grid(data, chunk)
    # the corpus is raw throughout this stretch at 64-byte chunks: alternate compressible (zero) and random chunks
    # across the 1024-tile line, so that packages of both kinds sit on both sides of it
    line = 1024 * TILE
    window = list(range(line - 8, line + 8))
    for i in window[0::2]:
        data[i * chunk:(i + 1) * chunk] = 0
    _noise(data, chunk, window[1::2], 730)
    grid.patch(window)
    for side in (grid.types[line - 8:line], grid.types[line:line + 8]):
        assert (side == 255).any() and (side != 255).any()
    want = grid.expect(True)
    _run_both(eng, data, chunk, True, want, "chunk 64")
