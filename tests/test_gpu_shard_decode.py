"""Sharded decode of one body, simulated on one GPU: R ranks each get a copy of their own byte range of the
body (plus the header halo), run the range index (ambc_range_index), the fold in rank order
(ambc_range_fold), fetch the payload tail their last decoded package needs from the next ranks, list their
table (ambc_range_table) and decode their output slice.  For every body and split the result must be the
single-GPU walk's: the same outcome as ambc_index_dev (marker mismatch or covered bytes), the same table
once mapped back to global offsets with adjacent raw pieces merged, and the same output and status as
engine.decompress_device and the oracle."""
import bz2
import lzma
import zlib

import numpy as np
import pytest

import inputs
import oracle as O

pytestmark = pytest.mark.gpu

MARKER = b"\xff\xff\x00\x00"
WORLDS = (1, 2, 3, 5, 8, 17)
DT = np.dtype([("src_off", "<u8"), ("dst_off", "<u8"), ("comp_len", "<u4"), ("orig_len", "<u4"), ("type", "<u4"),
               ("out_len", "<u4")])


@pytest.fixture(scope="module")
def eng():
    from adaptive_compression_b200 import engine
    engine.require_cuda()
    return engine


def _dev(b):
    import torch
    a = np.frombuffer(bytes(b), dtype=np.uint8)
    return torch.from_numpy(a.copy()).to("cuda") if a.size else torch.empty(0, dtype=torch.uint8, device="cuda")


def _rows(t_table, n):
    return [tuple(int(e[k]) for k in DT.names) for e in t_table.cpu().numpy()[:n * 32].view(DT)]


def _merge(rows):
    """adjacent raw pieces (contiguous in body and output) -> one entry"""
    out = []
    for r in rows:
        if out and r[4] == 255 and out[-1][4] == 255 and r[0] == out[-1][0] + out[-1][5] and r[1] == out[-1][1] + out[-1][5]:
            p = out[-1]
            out[-1] = (p[0], p[1], p[2] + r[2], p[3] + r[3], 255, p[5] + r[5])
        else:
            out.append(r)
    return out


def simulate(eng, body, cuts, orig_size, marker=MARKER, known=None):
    """-> ('marker',) or ('ok', merged global table, covered, output bytes, summed status)"""
    import torch
    from adaptive_compression_b200 import _lib as L
    from adaptive_compression_b200 import distributed as D
    known = L.NATIVE_MASK if known is None else known
    Lb, mb = len(body), len(marker)
    ranges = list(zip(cuts[:-1], cuts[1:]))
    bufs, ris = [], []
    for lo, hi in ranges:
        b0, b1 = D.buffer_span(lo, hi, Lb, mb)
        bufs.append(_dev(body[b0:b1]))  # a copy: nothing outside the range and its halo is reachable
        ris.append(eng.range_index(bufs[-1], lo, hi, Lb, orig_size, marker, known))
    st, entries = eng.range_init_state(), []
    for ri in ris:
        entries.append(st)
        st = eng.range_fold(ri, st)
    if st.status == L.RANGE_MARKER:
        return ("marker",)
    covered = min(st.out_before, orig_size)
    slices = D.output_slices(entries, ranges, orig_size, mb, known)
    needs = [eng.range_table(ri, e, count_only=True)[4] for ri, e in zip(ris, entries)]
    for r, need in enumerate(needs):
        if need:
            bufs[r] = torch.cat([bufs[r], torch.zeros(need, dtype=torch.uint8, device="cuda")])
    for src, dst, g0, g1 in D.tail_fetch_plan(ranges, needs, Lb, mb):
        bufs[dst][g0 - ranges[dst][0]:g1 - ranges[dst][0]] = bufs[src][g0 - ranges[src][0]:g1 - ranges[src][0]]
    rows, outs, status = [], [], [0, 0]
    for r, (ri, e) in enumerate(zip(ris, entries)):
        t_table, n, olo, ohi, _ = eng.range_table(ri, e)
        o0, o1 = slices[r]
        assert olo == o0 and ohi == (slices[r + 1][0] if r + 1 < len(slices) else covered), (r, olo, ohi, slices)
        lo = ranges[r][0]
        rows += [(x[0] + lo, x[1] + o0) + x[2:] for x in _rows(t_table, n)]
        out, stt = eng.range_decode(bufs[r], t_table, n, o1 - o0, known)
        outs.append(out.cpu().numpy().tobytes())
        status = [status[0] + stt[0], status[1] + stt[1]]
    return ("ok", _merge(rows), covered, b"".join(outs), status)


def reference(eng, body, orig_size, marker=MARKER, known=None):
    from adaptive_compression_b200 import _lib as L
    known = L.NATIVE_MASK if known is None else known
    t = _dev(body)
    try:
        tt, ne, cov = eng.index_device(t, orig_size, marker, known)
    except ValueError as e:
        assert "Marker mismatch" in str(e)
        return ("marker",)
    out, st = eng.decompress_device(t, orig_size, marker, known)
    return ("ok", _merge(_rows(tt, ne)), cov, out.cpu().numpy().tobytes(), st)


def headers(body, mb=4):
    """header positions of the serial walk over a well-formed body"""
    pos, hs = 0, []
    while pos + mb + 14 <= len(body):
        hs.append(pos)
        if body[pos + mb] == 0:
            break
        pos += mb + 14 + int.from_bytes(body[pos + mb + 10:pos + mb + 14], "little")
    return hs


def splits(Lb, hs, seed, raw_spans=()):
    """rank cuts [0, ..., Lb]: even and random for every world size, exactly at headers, 1..21 bytes into
    headers, inside raw payloads, at Lb, and empty ranges"""
    rs = np.random.RandomState(seed)
    out = []
    for R in WORLDS:
        out.append([Lb * r // R for r in range(R + 1)])
        out.append([0] + sorted(int(x) for x in rs.randint(0, Lb + 1, R - 1)) + [Lb])
    inner = [h for h in hs if 0 < h < Lb]
    for d in range(0, 22):
        pts = sorted({min(h + d, Lb) for h in inner})
        if pts:
            pick = sorted(set(pts[int(i)] for i in np.linspace(0, len(pts) - 1, min(7, len(pts)))))
            out.append([0] + pick + [Lb])
    for a, b in raw_spans:
        if b - a > 2:
            out.append([0, a + 1, (a + b) // 2, b - 1, Lb])
    out += [[0, Lb, Lb, Lb], [0, 0, 0, Lb], [0, Lb // 2, Lb // 2, Lb, Lb]]
    return out


def check_all(eng, body, orig_size, seed, marker=MARKER, known=None, oracle=True, cuts=None, raw_spans=()):
    want = reference(eng, body, orig_size, marker, known)
    # the oracle only where the single-GPU decode reports no malformed package: on a stream whose decoded length
    # differs from its header (status[1]) the GPU decoders zero-fill the entry (include/ambc.h), while the
    # reference's Huffman decoder, for one, decodes the padding bits on up to the header's original_length
    if want[0] == "ok" and oracle and want[4] == [0, 0]:
        assert want[3] == O.decompress_body(bytes(body), orig_size, marker)
    for c in (cuts if cuts is not None else splits(len(body), headers(body, len(marker)), seed, raw_spans)):
        got = simulate(eng, body, c, orig_size, marker, known)
        if want[0] == "marker":
            assert got == want, (c, got[0])
            continue
        assert got[0] == "ok", (c, got[0])
        assert got[2] == want[2], (c, "covered", got[2], want[2])
        assert got[1] == want[1], (c, "table", len(got[1]), len(want[1]))
        assert got[3] == want[3], (c, "output")
        assert got[4] == want[4], (c, "status", got[4], want[4])
    return want


def pkg(t, orig, payload, marker=MARKER, comp=None):
    c = len(payload) if comp is None else comp
    return marker + bytes([t, 0]) + int(orig).to_bytes(4, "little") * 2 + int(c).to_bytes(4, "little") + payload


END = MARKER + b"\x00" * 12


def test_compressed_bodies_fixed(eng):
    from adaptive_compression_b200 import _lib as L
    for seed, n, chunk, kinds, flags in [(1, 1 << 20, 4096, 0b1011111, 0), (2, 600000, 1024, 0b1111111, 0),
                                         (3, 700000, 4096, 0b1111111, L.F_PER_CHUNK_RAW)]:
        t = eng.synth(n, seed * 65536, kind_mask=kinds)
        o = eng.compress_device(t, chunk, flags=flags)
        body = o.body.cpu().numpy().tobytes()
        hs = headers(body)
        raws = [(h + 18, h + 18 + int.from_bytes(body[h + 14:h + 18], "little")) for h in hs if body[h + 4] == 255]
        want = check_all(eng, body, n, seed, raw_spans=raws[:3])
        assert want[0] == "ok" and want[3] == t.cpu().numpy().tobytes()
        for osz in (0, 1, n // 3, n - 1, n + 777):
            check_all(eng, body, osz, seed, cuts=splits(len(body), hs, seed + osz)[::3])


def test_compressed_bodies_dynamic(eng):
    t = eng.synth(500000, 7 << 16, kind_mask=0b1111111)
    o = eng.compress_dynamic_device(t, [16384, 4096, 1024])
    body = o.body.cpu().numpy().tobytes()
    want = check_all(eng, body, 500000, 11)
    assert want[3] == t.cpu().numpy().tobytes()


def test_stdlib_codec_packages_and_tail_fetch(eng):
    """types 5-7 with payloads up to ~500 KB: a decoded package's payload runs over several ranges"""
    from adaptive_compression_b200 import _lib as L
    known = L.NATIVE_MASK | (1 << 5) | (1 << 6) | (1 << 7)
    a, b, c = inputs.rand(480000, 1), inputs.text(300000, 2), inputs.rand(200000, 3) + inputs.log(90000, 4)
    body = (pkg(1, 12, b"A\x06B\x06") + pkg(5, len(a), zlib.compress(a, 9)) + pkg(255, 7000, inputs.rand(7000, 5)) +
            pkg(6, len(b), bz2.compress(b)) + pkg(7, len(c), lzma.compress(c)) + pkg(2, 5, b"\x00a\x00b\x00c\x00d\x00e") + END)
    want_out = b"A" * 6 + b"B" * 6 + a + inputs.rand(7000, 5) + b + c + b"abcde"
    want = check_all(eng, body, len(want_out), 21, known=known, oracle=False)
    assert want[3] == want_out and want[4] == [0, 0]
    # the same body with only some codecs known: the others are copied through
    check_all(eng, body, len(want_out), 22, known=L.NATIVE_MASK | (1 << 6), oracle=False)


def test_damaged_bodies(eng):
    data = inputs.mixed_file(5, 2048, 77) + inputs.text(300, 78)
    body, pm = O.compress_body(data, 2048)
    bounds, pos = [], 0
    for t, orig, comp in pm:
        bounds.append(pos); pos += 18 + comp
    cuts = set()
    for b in bounds + [pos, len(body)]:
        for d in (-20, -5, -1, 0, 1, 3, 4, 5, 17, 18, 19, 40):
            if 0 <= b + d <= len(body):
                cuts.add(b + d)
    rs = np.random.RandomState(3)
    for i, cut in enumerate(sorted(cuts)):  # truncation at every boundary kind
        bb = body[:cut]
        check_all(eng, bb, len(data), i, cuts=[splits(len(bb), headers(bb), i)[k] for k in rs.randint(0, 12, 3)])
    for b in bounds[1:]:  # marker and length fields of every package
        for off in (0, 3, 4, 6, 10, 13, 14, 17):
            bad = bytearray(body); bad[b + off] ^= 0x5A
            check_all(eng, bytes(bad), len(data), b + off, cuts=splits(len(bad), bounds, b)[::4])


def test_odd_packages(eng):
    fake = MARKER + bytes([3, 0]) + (100).to_bytes(4, "little") * 2 + (7).to_bytes(4, "little")  # looks like a header
    raw1 = b"abc" + fake + b"xyz" * 10 + MARKER + MARKER
    body = pkg(255, len(raw1), raw1) + pkg(1, 12, b"A\x06B\x06") + pkg(9, 30, b"unknown-type-payload") + \
        pkg(255, 50, b"short raw, padded") + pkg(4, 10, b"") + pkg(2, 5, b"\x00a\x00b\x00c\x00d\x00e") + END
    every = [[0] + [k] + [len(body)] for k in range(len(body) + 1)]  # a two-rank cut at every byte
    for osz in (0, 10, len(raw1), len(raw1) + 12, 200, 1000):
        for known in (None, 0b110, 0b1111111110):
            check_all(eng, body, osz, osz, known=known, oracle=known is None)
    check_all(eng, body, 200, 0, cuts=every)
    for b in (pkg(1, 4, b"Z\x04") + END + pkg(1, 4, b"Y\x04") + END, END, b"", MARKER + b"\x01",
              b"\x00" + pkg(1, 4, b"Z\x04") + END, pkg(1, 4, b"Z\x04") + b"garbage-not-a-marker-but-long-enough",
              pkg(1, 4, b"Z\x04"), pkg(1, 4, b"Z\x04") + b"\xff\xff"):
        for osz in (0, 10, 100):
            check_all(eng, b, osz, len(b), cuts=[[0] + [k] + [len(b)] for k in range(len(b) + 1)] + [[0, len(b)]])
    for mk in (b"\xf8", b"\xab\xcd", b"\x01\x02\x03"):
        b2 = pkg(1, 4, b"Z\x04", marker=mk) + pkg(255, 6, b"qwerty" + mk, marker=mk) + mk + b"\x00" * 12
        for bb in (b2, b2[:-5]):
            check_all(eng, bb, 10, 1, marker=mk, oracle=False, cuts=[[0] + [k] + [len(bb)] for k in range(len(bb) + 1)])


def test_large_raw_package_over_many_ranks(eng):
    big = inputs.rand(300000, 9)
    body = pkg(1, 4, b"Z\x04") + pkg(255, len(big), big) + pkg(1, 4, b"Y\x04") + END
    for osz in (4 + len(big) + 4, 4 + 100000, 4 + len(big) + 4000):
        check_all(eng, body, osz, osz, raw_spans=[(40, 40 + len(big))])
    # a padded raw package (orig > comp) whose payload ends exactly at a range boundary
    short = pkg(255, 200000, big[:70000]) + pkg(1, 4, b"Y\x04") + END
    check_all(eng, short, 200004, 5, cuts=[[0, 18 + 70000, len(short)], [0, 17 + 70000, 19 + 70000, len(short)],
                                            [0, 30000, 60000, 18 + 70000, 18 + 70000, len(short)]])
