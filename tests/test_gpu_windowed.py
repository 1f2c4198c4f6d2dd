"""The windowed file -> file paths (windowed.py, DESIGN.md §4.6) against the in-memory paths, the oracle and the
golden files: windows down to one chunk or one segment, so that every case crosses many window boundaries."""
import hashlib
import os

import numpy as np
import pytest

import inputs
import oracle as O

pytestmark = pytest.mark.gpu

STAT_KEYS = ("original_size", "compressed_size", "ratio", "percent_reduction", "chunk_stats", "overhead_bytes",
             "compression_efficiency")


@pytest.fixture(scope="module")
def eng():
    from adaptive_compression_b200 import engine
    engine.require_cuda()
    return engine


def _window(monkeypatch, W):
    from adaptive_compression_b200 import adaptive_compressor as A
    monkeypatch.setattr(A, "window_bytes", lambda need, device_bytes: W)


def _make(cfg):
    from adaptive_compression_b200 import AdaptiveCompressor
    return AdaptiveCompressor(chunk_size=cfg["chunk_size"], methods=cfg.get("method_ids"),
                              per_chunk_raw=bool(cfg.get("per_chunk_raw")),
                              use_marker_search=bool(cfg.get("found_marker")))


def both(tmp_path, monkeypatch, data, cfg, windows, decode=True):
    """compress (and decompress) with the in-memory facade and with every window size: identical files and stats"""
    src, ref = tmp_path / "in.bin", tmp_path / "ref.ambc"
    src.write_bytes(data)
    _window(monkeypatch, None)
    want_stats = _make(cfg).compress(str(src), str(ref))
    want = ref.read_bytes()
    for W in windows:
        _window(monkeypatch, W)
        dst, back = tmp_path / ("w%d.ambc" % W), tmp_path / ("w%d.out" % W)
        c = _make(cfg)
        stats = c.compress(str(src), str(dst))
        got = dst.read_bytes()
        assert got == want, (cfg, W, len(got), len(want))
        for k in STAT_KEYS:
            assert stats[k] == want_stats[k], (cfg, W, k, stats[k], want_stats[k])
        if decode and got[:4] == b"AMBC":
            c.decompress(str(dst), str(back))
            assert back.read_bytes() == data, (cfg, W)
            assert c.last_status == [0, 0]
        dst.unlink()
    if want[:4] == b"AMBC":
        assert O.decompress_file(want, known=tuple(cfg.get("method_ids") or (1, 2, 3, 4)) + (255,)) == data
    return want


def _windows(n, unit):
    return sorted({unit, 7 * unit, 7 * unit + unit // 3, max(unit, n), 2 * n + unit})


def test_fixed_grid_files(tmp_path, monkeypatch, eng):
    for chunk in (4096, 8192, 3000):
        data = inputs.mixed_file(40, chunk, chunk) + inputs.text(1234, 5)
        both(tmp_path, monkeypatch, data, {"chunk_size": chunk}, _windows(len(data), chunk))
    for name, data, cfg in inputs.container_cases():
        both(tmp_path, monkeypatch, data, cfg, _windows(len(data), cfg["chunk_size"]))


def test_fixed_grid_synthetic_corpus(tmp_path, monkeypatch, eng):
    n = (24 << 20) + 777
    data = eng.synth(n, 5 << 20, kind_mask=0b1011111).cpu().numpy().tobytes()
    both(tmp_path, monkeypatch, data, {"chunk_size": 4096}, (4096 * 61, 1 << 20, 3 << 20))


def test_raw_tail_in_every_position(tmp_path, monkeypatch, eng):
    chunk, k = 4096, 5  # 5 chunks per window
    for at in (0, 2, 4, 5, 9, 14, 20, 24):
        data = bytearray(inputs.mixed_file(25, chunk, 70 + at, ("text", "log", "runs")))
        data[at * chunk:(at + 1) * chunk] = inputs.rand(chunk, at)
        for pcr in (False, True):
            both(tmp_path, monkeypatch, bytes(data), {"chunk_size": chunk, "per_chunk_raw": pcr}, (k * chunk, chunk))


def test_verbatim_store(tmp_path, monkeypatch, eng):
    data = inputs.rand(300000, 4)
    got = both(tmp_path, monkeypatch, data, {"chunk_size": 4096}, (4096, 65536))
    assert got == data


def test_compress_error_leaves_no_output(tmp_path, monkeypatch, eng):
    """an error inside a windowed compress (candidates whose gcd the chain walk cannot grid): the output file is
    left as it was and no temporary file remains; through a symlink, the link stays and its target is replaced"""
    from adaptive_compression_b200 import AdaptiveCompressor
    from adaptive_compression_b200._lib import AmbcError
    src, dst = tmp_path / "in.bin", tmp_path / "out.ambc"
    data = inputs.mixed_file(20, 4096, 5, ("text", "log"))
    src.write_bytes(data)
    dst.write_bytes(b"keep")
    _window(monkeypatch, 65536)
    c = AdaptiveCompressor()
    c.CHUNK_SIZE_CANDIDATES = [4096, 1000]
    with pytest.raises(AmbcError):
        c.compress(str(src), str(dst))
    assert dst.read_bytes() == b"keep" and sorted(os.listdir(tmp_path)) == ["in.bin", "out.ambc"]
    (tmp_path / "link.ambc").symlink_to(dst)
    AdaptiveCompressor(chunk_size=4096).compress(str(src), str(tmp_path / "link.ambc"))
    assert os.path.islink(tmp_path / "link.ambc") and dst.read_bytes() == O.compress_file(data, 4096)[0]


def test_multi_candidate_mode(tmp_path, monkeypatch, eng, golden):
    from adaptive_compression_b200 import distributed as D
    cases = {c[0]: c for c in inputs.dynamic_cases()}
    for row in golden["container_dyn_kat"]:
        name, data, cfg = cases[row["name"]]
        seg = D.DYN_SEGU * D._gcd_of(cfg["chunk_size"])
        got = both(tmp_path, monkeypatch, data, row["cfg"], (seg, 2 * seg, 5 * seg))
        assert hashlib.sha256(got).hexdigest() == row["ambc_sha256"], name
    # the cascade of DESIGN §4.3 (runs, then log lines) across windows, and a stop in a middle window
    casc = inputs.runs(150000, 8, max_run=5000) + inputs.log(150000, 9)
    stop = bytearray(inputs.mixed_file(30, 4096, 12, ("text", "log")))
    stop[61000:75000] = inputs.rand(14000, 2)
    for cands in (inputs.REF_DEFAULT_CANDIDATES, (8192, 4096), (1280, 768, 512)):
        seg = D.DYN_SEGU * D._gcd_of(cands)
        for data in (casc, bytes(stop)):
            want = both(tmp_path, monkeypatch, data, {"chunk_size": list(cands)}, (seg, 2 * seg, 5 * seg))
            assert want == O.compress_file(data, cands)[0]


def test_marker_search_carry_across_windows(tmp_path, monkeypatch, eng):
    """random bytes hold every 16-bit value; v0 = the marker of the bytes (the smallest absent value of more than 16
    bits) is written across a window boundary, so it occurs only there: without the carry bits the search would
    pick it"""
    from adaptive_compression_b200 import windowed
    W = 1 << 16
    r = bytearray(inputs.rand(1 << 20, 91))
    v0, bits = O.find_marker(bytes(r))
    assert bits > 16
    r[W - 1:W - 1 + len(v0)] = v0
    data = bytes(r)
    want = O.find_marker(data)
    assert want != (v0, bits)
    src = tmp_path / "m.bin"
    src.write_bytes(data)
    for w in (W, 3 * W):
        assert windowed.find_marker(str(src), len(data), w) == want
    both(tmp_path, monkeypatch, data[:300000], {"chunk_size": 4096, "found_marker": True}, (W,), decode=False)
    for name, d, max_len, sample in inputs.marker_cases():
        if sample:
            continue
        src.write_bytes(d)
        try:
            want = O.find_marker(d, max_len)
        except ValueError:
            with pytest.raises(ValueError):
                windowed.find_marker(str(src), len(d), 4096, max_len)
            continue
        for w in (1, 7, 4096):
            assert windowed.find_marker(str(src), len(d), w, max_len) == want, (name, w)


# ---- decompress ------------------------------------------------------------------------------------------------
def _headers(body, mb=4):
    pos, hs = 0, []
    while pos + mb + 14 <= len(body):
        hs.append(pos)
        if body[pos + mb] == 0:
            break
        pos += mb + 14 + int.from_bytes(body[pos + mb + 10:pos + mb + 14], "little")
    return hs


def _decode(tmp_path, body, orig, W, budget=None, known=None, marker=b"\xff\xff\x00\x00"):
    from adaptive_compression_b200 import _lib as L
    from adaptive_compression_b200 import windowed
    p, q = tmp_path / "body.bin", tmp_path / "body.out"
    p.write_bytes(b"HDR" + body)
    with open(q, "wb") as f:
        md5, status = windowed.decompress(str(p), f, 3, len(body), orig, W, marker,
                                          L.NATIVE_MASK if known is None else known, budget)
    out = q.read_bytes()
    assert hashlib.md5(out).digest() == md5
    return out, status


def _reference(eng, body, orig, known=None, marker=b"\xff\xff\x00\x00"):
    from adaptive_compression_b200 import _lib as L
    t = eng.to_device(body)
    try:
        out, st = eng.decompress_device(t, orig, marker, L.NATIVE_MASK if known is None else known)
    except ValueError:
        return None
    return out.cpu().numpy().tobytes(), st


def _cuts(body):
    hs = [h for h in _headers(body) if h > 0]
    Ws = {1 << 12, 1 << 16, len(body), len(body) + 5}
    for d in (0, 1, 5, 13, 17, 21):
        for h in hs[:3] + hs[-2:]:
            Ws.add(h + d)
    return sorted(w for w in Ws if w > 0)


def check_decode(tmp_path, eng, body, orig, known=None, budget=None, Ws=None):
    want = _reference(eng, body, orig, known)
    for W in (Ws or _cuts(body)):
        if want is None:
            with pytest.raises(ValueError, match="Marker mismatch in chunk header."):
                _decode(tmp_path, body, orig, W, budget, known)
            continue
        out, st = _decode(tmp_path, body, orig, W, budget, known)
        assert out == want[0], (W, len(out), len(want[0]))
        assert st == want[1], (W, st, want[1])
    return want


def test_decode_compressed_bodies(tmp_path, eng):
    for seed, n, chunk, flags in [(1, 600000, 4096, 0), (2, 300000, 3000, 1)]:
        t = eng.synth(n, seed << 16, kind_mask=0b1111111)
        o = eng.compress_device(t, chunk, flags=flags)
        body = o.body.cpu().numpy().tobytes()
        assert check_decode(tmp_path, eng, body, n)[0] == t.cpu().numpy().tobytes()
        for osz in (0, n // 3, n + 777):
            check_decode(tmp_path, eng, body, osz, Ws=_cuts(body)[::3])
    t = eng.synth(400000, 7 << 16, kind_mask=0b1111111)
    o = eng.compress_dynamic_device(t, [16384, 4096, 1024])
    check_decode(tmp_path, eng, o.body.cpu().numpy().tobytes(), 400000)


def _pkg(t, orig, payload, comp=None, marker=b"\xff\xff\x00\x00"):
    c = len(payload) if comp is None else comp
    return marker + bytes([t, 0]) + int(orig).to_bytes(4, "little") * 2 + int(c).to_bytes(4, "little") + payload


def test_decode_stdlib_packages_larger_than_the_window(tmp_path, eng):
    import bz2
    import lzma
    import zlib
    from adaptive_compression_b200 import _lib as L
    a, b, c = inputs.rand(480000, 1), inputs.text(300000, 2), inputs.rand(200000, 3) + inputs.log(90000, 4)
    END = b"\xff\xff\x00\x00" + bytes(12)
    body = (_pkg(1, 12, b"A\x06B\x06") + _pkg(5, len(a), zlib.compress(a, 9)) + _pkg(255, 7000, inputs.rand(7000, 5)) +
            _pkg(6, len(b), bz2.compress(b)) + _pkg(7, len(c), lzma.compress(c)) + _pkg(2, 5, b"\x00a\x00b\x00c\x00d\x00e") +
            END)
    for known in (L.NATIVE_MASK | (1 << 5) | (1 << 6) | (1 << 7), L.NATIVE_MASK | (1 << 6), L.NATIVE_MASK):
        check_decode(tmp_path, eng, body, 6 + 6 + len(a) + 7000 + len(b) + len(c) + 5, known=known, budget=65536,
                     Ws=(4096, 50000, 65536, len(body)))


def test_decode_damaged_bodies(tmp_path, eng):
    data = inputs.mixed_file(8, 2048, 77, ("text", "log", "runs")) + inputs.text(300, 78)
    body, pm = O.compress_body(data, 2048)
    hs = _headers(body)
    for cut in (hs[3], hs[3] + 5, hs[5] + 18, len(body) - 16, len(body) - 1):
        check_decode(tmp_path, eng, body[:cut], len(data), Ws=(2048, 5000, len(body)))
    for h in hs[1:6]:
        for off in (0, 3, 4, 10, 14):
            bad = bytearray(body)
            bad[h + off] ^= 0x5A
            check_decode(tmp_path, eng, bytes(bad), len(data), Ws=(1024, 4096, hs[2] + 3))


def test_decode_run_heavy_file_in_small_output_pieces(tmp_path, eng):
    """one repeated byte: ~80x at chunk 4096; the output budget is far below one window's output"""
    data = b"\x07" * (24 << 20)
    o = eng.compress_device(eng.to_device(data), 4096)
    body = o.body.cpu().numpy().tobytes()
    assert len(data) / len(body) > 70
    for W, budget in ((16384, 65536), (1 << 20, 1 << 18), (len(body), 1 << 20)):
        out, st = _decode(tmp_path, body, len(data), W, budget)
        assert out == data and st == [0, 0]


def test_facade_errors(tmp_path, monkeypatch, eng):
    data = inputs.mixed_file(12, 4096, 11, ("text", "log", "runs", "csv"))
    src, dst, back = tmp_path / "a", tmp_path / "a.ambc", tmp_path / "b"
    src.write_bytes(data)
    _window(monkeypatch, 4096)
    from adaptive_compression_b200 import AdaptiveCompressor
    c = AdaptiveCompressor(chunk_size=4096)
    c.compress(str(src), str(dst))
    good = dst.read_bytes()
    back.write_bytes(b"old")
    bad = bytearray(good); bad[0] = ord("X")
    dst.write_bytes(bad)
    with pytest.raises(ValueError, match="Magic mismatch"):
        c.decompress(str(dst), str(back))
    hs = _headers(good[47:])
    bad = bytearray(good); bad[47 + hs[5]] ^= 1
    dst.write_bytes(bad)
    with pytest.raises(ValueError, match="Marker mismatch in chunk header."):
        c.decompress(str(dst), str(back))
    assert back.read_bytes() == b"old"
    assert sorted(os.listdir(tmp_path)) == ["a", "a.ambc", "b"]
    bad = bytearray(good); bad[47 + 18 + 30] ^= 0x55
    dst.write_bytes(bad)
    _window(monkeypatch, None)
    mem = AdaptiveCompressor(chunk_size=4096)
    with pytest.raises(ValueError, match="Checksum mismatch"):
        mem.decompress(str(dst), str(back))
    want_out = back.read_bytes()
    _window(monkeypatch, 4096)
    with pytest.raises(ValueError, match="Checksum mismatch"):
        c.decompress(str(dst), str(back))
    assert back.read_bytes() == want_out and c.last_status == mem.last_status


def test_facade_and_cli(tmp_path, monkeypatch, eng):
    import sys
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, ROOT)
    import main
    from adaptive_compression_b200 import adaptive_compressor as A
    data = inputs.mixed_file(30, 4096, 21) + inputs.text(500, 22)
    src = tmp_path / "in.csv"
    src.write_bytes(data)
    outs = {}
    for W in (None, 65536):
        _window(monkeypatch, W)
        for args in (["--chunk-size", "4096"], []):
            dst, back = tmp_path / "o.ambc", tmp_path / "b.csv"
            main.main(["compress", str(src), str(dst), "--no-history"] + args)
            main.main(["decompress", str(dst), str(back)])
            assert back.read_bytes() == data
            outs.setdefault(tuple(args), set()).add(dst.read_bytes())
    assert all(len(v) == 1 for v in outs.values())
    # without the patch a small file takes the in-memory path
    monkeypatch.undo()
    assert A.window_bytes(1 << 20, lambda w: w) is None


def test_device_memory_is_bounded_by_the_window(tmp_path, eng):
    """the same W = 4 MiB for a 64 MiB and a 256 MiB file: the same peak of torch-allocated device memory, within
    the formulas of DESIGN §4.6"""
    import torch
    from adaptive_compression_b200 import _lib as L
    from adaptive_compression_b200 import windowed
    W = 4 << 20
    peaks = {}
    for n in (64 << 20, 256 << 20):
        src = tmp_path / "s.bin"
        eng.synth(n, 0, kind_mask=0b1011111).cpu().numpy().tofile(str(src))
        for kind in ("fixed", "dynamic", "decompress"):
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            with open(tmp_path / "s.out", "wb") as f:
                if kind == "fixed":
                    body_len = windowed.compress_fixed(str(src), f, n, 4096, W)[0]
                elif kind == "dynamic":
                    windowed.compress_dynamic(str(src), f, n, inputs.REF_DEFAULT_CANDIDATES, W)
                else:
                    windowed.decompress(str(tmp_path / "s.body"), f, 0, body_len, n, W)
            if kind == "fixed":
                os.replace(tmp_path / "s.out", tmp_path / "s.body")
            peaks[(kind, n)] = torch.cuda.max_memory_allocated() - base
        if n == 256 << 20:
            back = np.fromfile(str(tmp_path / "s.out"), dtype=np.uint8)
            assert np.array_equal(back, np.fromfile(str(src), dtype=np.uint8))
    bounds = {"fixed": windowed.fixed_device_bytes(W, 4096), "dynamic": windowed.dynamic_device_bytes(W, inputs.REF_DEFAULT_CANDIDATES),
              "decompress": windowed.decompress_device_bytes(W, W, n_cand=W // 18 + 64)}
    slack = 1 << 20  # status words, method maps, the allocator's 512-byte rounding
    for kind, bound in bounds.items():
        a, b = peaks[(kind, 64 << 20)], peaks[(kind, 256 << 20)]
        assert abs(a - b) <= slack, (kind, a, b)
        assert max(a, b) <= bound + slack, (kind, a, b, bound)
    assert L.NATIVE_MASK
