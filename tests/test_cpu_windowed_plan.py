"""The host side of windowed.py.  The window assembly restated over the oracle (as test_cpu_dynamic_shard.py does for
ranks): every window's oracle body, or the packages of the oracle's chunk chain that start in it, framed and encoded
one by one with the oracle's codecs, go through windowed.window_parts; with the END package behind the last window
the result must be oracle.compress_file's body of the whole input, for 1-24 windows and raw tails in every position.
Also: the 4 GiB refusal, the cut of a decode table into output pieces (out_len up to 2^32 - 1), and the temporary
file the windowed facade writes before its rename."""
import os
import stat
import struct

import numpy as np
import pytest
import torch

import inputs
import oracle as O
from adaptive_compression_b200 import distributed as D
from adaptive_compression_b200 import windowed as Wd

MARKER = b"\xff\xff\x00\x00"


def _assemble(parts_of_windows, n):
    out = bytearray()
    for parts, body, data in parts_of_windows:
        for p in parts:
            out += p if isinstance(p, bytes) else (body if p[0] == "body" else data)[p[1]:p[2]]
    return bytes(out) + D.end_package(MARKER)


def fixed_plan(data, chunk, W, pcr):
    n, raw, wins = len(data), False, []
    for lo, hi in Wd.fixed_windows(n, chunk, W):
        win = data[lo:hi]
        if raw:
            wins.append(([("input", 0, hi - lo)], b"", win))
            continue
        body, pm = O.compress_body(win, chunk, per_chunk_raw=pcr)
        fr = next((i for i, p in enumerate(pm) if p[0] == 255), -1) if not pcr else -1
        raw_at = lo + fr * chunk if fr >= 0 else None
        wins.append((Wd.window_parts(D.packed_bytes(len(body), hi - lo, fr, chunk), raw_at, lo, hi, n, MARKER), body, win))
        raw = raw_at is not None
    return _assemble(wins, n)


def _package(t, chunk):
    payload = O.compress(t, chunk, lz_fast=True)
    return MARKER + bytes([t, 0]) + struct.pack("<III", len(chunk), len(chunk), len(payload)) + payload


def dyn_plan(data, cands, W):
    """each window's fragment = the packages of the chunk chain (the oracle's package list: the positions and methods
    the range walk, resolve and encode find) whose chunk starts in it, each framed and encoded on its own; the chain
    stops at the first raw package"""
    n = len(data)
    _, pm = O.compress_body(data, cands)
    chain, pos = [], 0
    for t, orig, _ in pm:
        chain.append((pos, t, orig))
        pos += orig
    wins, raw = [], False
    for lo, hi in Wd.dyn_windows(n, cands, W):
        if raw:
            wins.append(([("input", 0, hi - lo)], b"", data[lo:hi]))
            continue
        mine = [c for c in chain if lo <= c[0] < hi]
        stop = next((p for p, t, _ in mine if t == 255), None)
        frag = b"".join(_package(t, data[p:p + orig]) for p, t, orig in mine if p != stop)
        wins.append((Wd.window_parts(len(frag), stop, lo, hi, n, MARKER), frag, data[lo:hi]))
        raw = stop is not None
    return _assemble(wins, n)


def _with_random_chunk(chunk, n_chunks, at, seed):
    """a mixed file whose chunk `at` (None: none) has no winner"""
    data = bytearray(inputs.mixed_file(n_chunks, chunk, seed, ("text", "log", "runs", "csv")))
    if at is not None:
        data[at * chunk:(at + 1) * chunk] = inputs.rand(chunk, seed + 1)
    return bytes(data)


def test_fixed_grid_windows_equal_the_whole_file():
    bad = []
    for chunk in (4096, 3000):
        n_chunks = 23
        for at in (None, 0, 1, 6, 7, 13, 21, 22):
            data = _with_random_chunk(chunk, n_chunks, at, 40 + (at or 0)) + inputs.text(777, 3)
            for pcr in (False, True):
                want = O.compress_body(data, chunk, per_chunk_raw=pcr)[0]
                for k in (1, 2, 3, 5, 7, 11, 20, 24):  # chunks per window: 24 windows down to one
                    got = fixed_plan(data, chunk, k * chunk + (chunk // 3 if k % 2 else 0), pcr)
                    if got != want:
                        bad.append((chunk, at, pcr, k))
    assert not bad, bad


def test_fixed_grid_file_matches_oracle_file():
    data = _with_random_chunk(4096, 12, 5, 9)
    ambc, stored, _ = O.compress_file(data, 4096)
    assert not stored
    hs = len(ambc) - len(O.compress_body(data, 4096)[0])
    for W in (4096, 3 * 4096, 1 << 20):
        assert fixed_plan(data, 4096, W, False) == ambc[hs:]


def test_multi_candidate_windows_equal_the_whole_file():
    bad = []
    rs = np.random.RandomState(5)
    for cands in ((8192, 4096), (1280, 768, 512)):
        seg = D.DYN_SEGU * D._gcd_of(cands)
        for trial in range(6):
            n_seg = int(rs.randint(2, 21))
            data = bytearray(inputs.mixed_file(n_seg * seg // 4096 + 1, 4096, 60 + trial, ("text", "log", "runs")))
            data = data[:n_seg * seg - int(rs.randint(0, seg // 2))]
            if trial % 2:  # a stretch without any winner: the chain stops there
                at = int(rs.randint(0, len(data) - 9000))
                data[at:at + 9000] = inputs.rand(9000, trial)
            data = bytes(data)
            want = O.compress_body(data, cands)[0]
            for k in (1, 2, 5, 20):
                if dyn_plan(data, cands, k * seg) != want:
                    bad.append((cands, trial, k))
    assert not bad, bad


def test_raw_package_of_4_gib_is_refused_before_the_window_is_written():
    n = (4 << 30) + 4096
    with pytest.raises(struct.error, match="'I' format requires 0 <= number <= 4294967295"):
        Wd.window_parts(100, 0, 0, 4096, n, MARKER)
    at = n - 0xFFFFFFFF  # the longest raw package there is
    assert Wd.window_parts(100, at, 0, at + 10, n, MARKER)[1:] == [D.raw_package_header(MARKER, 0xFFFFFFFF),
                                                                  ("input", at, at + 10)]
    from adaptive_compression_b200 import _lib as L
    with pytest.raises(L.AmbcError):
        D.refuse_dyn_raw(n, 0)
    D.refuse_dyn_raw(n, at)


DT = np.dtype([("src_off", "<u8"), ("dst_off", "<u8"), ("comp_len", "<u4"), ("orig_len", "<u4"), ("type", "<u4"),
               ("out_len", "<u4")])


def _table(out_lens, start=0):
    t = np.zeros(len(out_lens), DT)
    t["out_len"] = out_lens
    t["dst_off"] = start + np.concatenate([[0], np.cumsum(np.array(out_lens, dtype=np.uint64))[:-1]])
    t["type"] = 255
    return torch.from_numpy(t.view(np.uint8).copy())


def test_decode_pieces_cut_with_large_out_len():
    """entries that claim 2^31 bytes or more (a raw tail of 2-4 GiB, a type 5-7 package) keep their unsigned
    length: every piece covers its entries exactly, stays within the budget unless it is one entry, and the pieces
    tile the window's output"""
    rs = np.random.RandomState(1)
    for case in range(40):
        k = int(rs.randint(1, 30))
        lens = [int(x) for x in rs.randint(0, 70000, k)]
        for at in rs.randint(0, k, int(rs.randint(0, 3))):
            lens[at] = int(rs.choice([1 << 31, 3_000_000_000, 0xFFFFFFFF]))
        start = int(rs.randint(0, 2)) * 17
        tt = _table(lens, start)
        w, ends = Wd.table_words(tt, k)
        assert ends.tolist() == [start + sum(lens[:i + 1]) for i in range(k)]
        budget = int(rs.choice([1, 4096, 65536, 1 << 20]))
        cuts = Wd.piece_cuts(w[:, 1], ends, budget)
        assert cuts[0][0] == 0 and cuts[0][2] == 0 and cuts[-1][1] == k and cuts[-1][3] == start + sum(lens)
        for (i, j, a, b), nxt in zip(cuts, cuts[1:] + [None]):
            assert j > i and b >= a
            assert b - a <= budget or j == i + 1 or (i == 0 and j == 1 + sum(1 for x in lens[1:j] if x == 0)), case
            assert int(w[i, 1]) >= a and int(ends[j - 1]) <= b
            if nxt is not None:
                assert nxt[0] == j and nxt[2] == b


def test_decode_pieces_run_through_a_fake_decoder():
    """_decode_pieces with range_decode replaced: every entry's bytes land at its output offset, the rest is zeros"""
    lens = [5, 300, 0, 7000, 40, 65536, 3]
    tt = _table(lens)
    span = sum(lens) + 123
    want = b"".join(bytes([1 + i]) * n for i, n in enumerate(lens)) + bytes(123)

    class Sink:
        def __init__(self):
            self.out = bytearray()

        def device(self, t):
            self.out += t.numpy().tobytes()

        def zeros(self, m):
            self.out += bytes(m)

    def fake_decode(buf, t_table, n, out_len, km, out=None):
        o = torch.zeros(out_len, dtype=torch.uint8)
        w, ends = Wd.table_words(t_table, n)
        for e in range(n):
            a, b = int(w[e, 1]), int(ends[e])
            assert 0 <= a <= b <= out_len
            o[a:b] = int(w[e, 3] & 0xFF)
        return o, [0, 0]
    tt.view(torch.int64).view(len(lens), 4)[:, 3] = \
        torch.tensor([(1 + i) | (n << 32) for i, n in enumerate(lens)], dtype=torch.int64)
    real = Wd.engine.range_decode
    try:
        Wd.engine.range_decode = fake_decode
        for budget in (1, 300, 5000, 1 << 20):
            sink = Sink()
            Wd._decode_pieces(None, tt.clone(), len(lens), span, budget, 0, sink, torch.empty(span, dtype=torch.uint8),
                              [0, 0])
            assert bytes(sink.out) == want, budget
    finally:
        Wd.engine.range_decode = real


def test_temporary_output_file(tmp_path):
    from adaptive_compression_b200 import adaptive_compressor as A
    old = os.umask(0o027)
    try:
        tmp, target = A._temp_beside(str(tmp_path / "new.ambc"))
        assert target == str(tmp_path / "new.ambc") and os.path.dirname(tmp) == str(tmp_path)
        assert stat.S_IMODE(os.stat(tmp).st_mode) == 0o640 and os.path.getsize(tmp) == 0
        os.unlink(tmp)
    finally:
        os.umask(old)
    real = tmp_path / "real.ambc"
    real.write_bytes(b"old")
    os.chmod(real, 0o604)
    (tmp_path / "link.ambc").symlink_to(real)
    tmp, target = A._temp_beside(str(tmp_path / "link.ambc"))
    assert target == str(real) and stat.S_IMODE(os.stat(tmp).st_mode) == 0o604
    os.replace(tmp, target)
    assert os.path.islink(tmp_path / "link.ambc") and real.read_bytes() == b""
