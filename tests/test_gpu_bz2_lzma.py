"""GPU tests of method ids 6 (BZip2Compression) and 7 (LZMACompression), where the reference calls the stdlib's bz2 and
lzma.  The oracles are stock bz2.decompress / lzma.decompress themselves: on every payload the GPU output equals what
the stock call returns, padded / truncated to original_length, or original_length zero bytes where it raises."""
import bz2
import hashlib
import lzma
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

import inputs

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MARKER = b"\xff\xff\x00\x00"


@pytest.fixture(scope="module")
def eng():
    from adaptive_compression_b200 import engine
    engine.require_cuda()
    return engine


def _stock(mod, payload, orig):
    try:
        out = mod.decompress(payload)
    except (OSError, ValueError, EOFError, lzma.LZMAError):
        return bytes(orig)
    return out[:orig].ljust(orig, b"\0")


def _check(eng, method, mod, payloads, origs):
    got = eng.codec_decode_batch(method, payloads, origs)
    bad = [(i, len(payloads[i]), origs[i]) for i, (g, p, o) in enumerate(zip(got, payloads, origs)) if g != _stock(mod, p, o)]
    assert not bad, bad[:10]


def _datas():
    r = np.random.RandomState(66)
    out = [inputs.make(k, n, 300 + n) for k in sorted(inputs.KINDS) for n in (1, 100, 4096, 8192, 131072, 262144)]
    out.append(bytes(262144))
    out.append(bytes(r.randint(0, 256, size=100000).astype(np.uint8)))
    return out


def _three(payload, n):
    """original_length equal, shorter and longer than the data"""
    return [(payload, n), (payload, max(1, n - 5)), (payload, n + 7)]


def test_bzip2_vs_stock(eng):
    datas = _datas()
    cases = []
    for d in datas:
        for level in (1, 9):
            cases += _three(bz2.compress(d, level), len(d))
    big = inputs.make("text", 300000, 3)  # several blocks at level 1
    cases += _three(bz2.compress(big, 1), len(big))
    two = bz2.compress(datas[3], 9) + bz2.compress(datas[10], 1)  # two concatenated streams
    cases += _three(two, len(datas[3]) + len(datas[10]))
    _check(eng, 6, bz2, [c for c, _ in cases], [o for _, o in cases])


def _bz2_crc(data):
    crc = 0xFFFFFFFF
    for ch in data:
        c = ((crc >> 24) ^ ch) << 24
        for _ in range(8):
            c = ((c << 1) ^ 0x04C11DB7) if c & 0x80000000 else (c << 1)
        crc = ((crc << 8) ^ c) & 0xFFFFFFFF
    return crc ^ 0xFFFFFFFF


def _randomised_stream(data):
    """a valid one-block stream with the `randomised` bit set (current bzip2 never writes one): the bit is set in a
    stock stream, stock libbzip2 says what the block then decodes to, and both CRCs are rewritten to match"""
    c = bytearray(bz2.compress(data, 9))
    c[14] ^= 0x80
    d = bz2.BZ2Decompressor()
    out = bytearray()
    try:
        out += d.decompress(bytes(c), max_length=1)
        while True:
            x = d.decompress(b"", max_length=1)
            if not x:
                break
            out += x
    except OSError:
        pass
    # the call that would return the last byte raises on the CRC instead: try every value of that byte
    old = int.from_bytes(c[10:14], "big")
    pad = next(p for p in range(8) if (int.from_bytes(c, "big") >> p) & ((1 << 80) - 1) == (0x177245385090 << 32) | old)
    for last in range(256):
        y = bytes(out) + bytes([last])
        new = _bz2_crc(y)
        v = int.from_bytes(c, "big") ^ ((old ^ new) << pad) ^ ((old ^ new) << (len(c) * 8 - 112))
        s = v.to_bytes(len(c), "big")
        try:
            if bz2.decompress(s) == y:
                return s, y
        except OSError:
            pass
    raise AssertionError("no randomised stream found")


def test_bzip2_randomised_blocks(eng):
    for n in (5000, 40000):
        data = inputs.make("text", n, 4)
        s, want = _randomised_stream(data)
        assert want != data  # the randomisation does change the block
        assert eng.codec_decode_batch(6, [s], [len(want)]) == [want]


def test_bzip2_errors_and_trailing_bytes(eng):
    d = inputs.make("csv", 20000, 5)
    c = bz2.compress(d, 9)
    cases = [c[:-1], c[:len(c) // 2], c[:4], b"BZh", c[:10] + bytes([c[10] ^ 1]) + c[11:],  # truncated, bad block CRC
             c[:-2] + bytes([c[-2] ^ 0x10]) + c[-1:],                                     # bad stream CRC
             b"BZh0" + c[4:], b"XZh9" + c[4:],
             c + b"junk", c + b"\0", c + b"B", c + b"BZh9", c + b"BZh91AY&SY", c + c[:-1], c + c + b"junk"]
    for p in cases[:8]:
        with pytest.raises((OSError, ValueError)):
            bz2.decompress(p)
    _check(eng, 6, bz2, cases, [len(d)] * len(cases))
    assert eng.codec_decode_batch(6, [b""], [10]) == [b""]


def _mutated(compress, seed, count):
    """valid streams with a flipped bit, a cut or an inserted byte (as test_gpu_inflate_mutated_streams_vs_zlib)"""
    r = np.random.RandomState(seed)
    kinds = sorted(inputs.KINDS)
    payloads, origs = [], []
    for i in range(count):
        d = inputs.make(kinds[i % len(kinds)], int(r.choice([200, 1500, 4096, 20000])), 15000 + i)
        c = bytearray(compress(d, r))
        what = r.randint(3)
        pos = int(r.randint(1, len(c)))  # (an empty payload is b'', the plug-in convention)
        if what == 0:
            c[pos] ^= 1 << int(r.randint(8))
        elif what == 1:
            del c[pos:]
        else:
            c.insert(pos, int(r.randint(256)))
        payloads.append(bytes(c))
        origs.append(len(d))
    return payloads, origs


def test_bzip2_mutated_streams_vs_stock(eng):
    p, o = _mutated(lambda d, r: bz2.compress(d, int(r.choice([1, 9]))), 616, 300)
    _check(eng, 6, bz2, p, o)


def test_lzma_vs_stock(eng):
    datas = _datas()
    cases = []
    for d in datas[::2]:
        for preset in (0, 6, 9, 9 | lzma.PRESET_EXTREME):
            cases += _three(lzma.compress(d, preset=preset), len(d))
    d = datas[4]
    for check in (lzma.CHECK_NONE, lzma.CHECK_CRC32, lzma.CHECK_CRC64):
        cases += _three(lzma.compress(d, check=check), len(d))
    for lc, lp, pb in ((0, 0, 0), (4, 0, 2), (0, 4, 4), (3, 1, 1), (1, 3, 0), (2, 2, 3)):
        cases.append((lzma.compress(d, filters=[{"id": lzma.FILTER_LZMA2, "preset": 6, "lc": lc, "lp": lp, "pb": pb}]), len(d)))
        cases.append((lzma.compress(d, format=lzma.FORMAT_ALONE,
                                    filters=[{"id": lzma.FILTER_LZMA1, "preset": 6, "lc": lc, "lp": lp, "pb": pb}]), len(d)))
    cases += _three(lzma.compress(d, filters=[{"id": lzma.FILTER_LZMA2, "preset": 9, "dict_size": 1 << 24}]), len(d))
    r = np.random.RandomState(7)
    noise = bytes(r.randint(0, 256, size=524288).astype(np.uint8))  # LZMA2 uncompressed chunks, many of them
    text = inputs.make("log", 524288, 9)
    small_noise = noise[:3000]
    cases += _three(lzma.compress(noise), len(noise)) + _three(lzma.compress(text), len(text))
    cases += _three(lzma.compress(small_noise), len(small_noise))
    cases += _three(lzma.compress(d) + lzma.compress(datas[6], check=lzma.CHECK_NONE), len(d) + len(datas[6]))
    cases.append((lzma.compress(d) + bytes(8) + lzma.compress(text), len(d) + len(text)))  # stream padding
    cases += _three(lzma.compress(d, format=lzma.FORMAT_ALONE), len(d))
    _check(eng, 7, lzma, [c for c, _ in cases], [o for _, o in cases])


def test_lzma_errors_and_trailing_bytes(eng):
    d = inputs.make("text", 20000, 6)
    x = lzma.compress(d)
    a = lzma.compress(d, format=lzma.FORMAT_ALONE)
    cases = [x[:-1], x[:len(x) // 2], x[:5], x[:-13] + bytes([x[-13] ^ 1]) + x[-12:],  # truncated, bad index CRC
             x[:12] + bytes([x[12] ^ 4]) + x[13:],                                      # bad block header
             x + b"\0" * 4, x + b"\xfd", x + b"\xfd7zXZ", a[:-3],
             lzma.compress(d, check=lzma.CHECK_SHA256),                                 # not implemented: an error
             x + b"junk", a + b"junk", x + b"\0" * 20, x + x + b"junk", x + x[:-1] + b"junk"]
    for p in cases[:9]:
        with pytest.raises(lzma.LZMAError):
            lzma.decompress(p)
    n_err = 10
    got = eng.codec_decode_batch(7, cases, [len(d)] * len(cases))
    assert got[n_err - 1] == bytes(len(d))  # SHA-256: zeros (documented gap)
    for i, (g, p) in enumerate(zip(got, cases)):
        if i != n_err - 1:
            assert g == _stock(lzma, p, len(d)), i
    assert eng.codec_decode_batch(7, [b""], [10]) == [b""]


def test_lzma_mutated_streams_vs_stock(eng):
    p, o = _mutated(lambda d, r: lzma.compress(d, preset=int(r.choice([0, 6]))), 717, 300)
    _check(eng, 7, lzma, p, o)


# ---- container -------------------------------------------------------------------------------------------------
def _body(seed):
    """packages of types 5, 6 and 7 with mixed sizes (18-byte headers, END package) -> (body, data, payload of pkg 0)"""
    import zlib
    r = np.random.RandomState(seed)
    kinds = sorted(inputs.KINDS)
    enc = {5: lambda c: zlib.compress(c, 9), 6: lambda c: bz2.compress(c, 9), 7: lambda c: lzma.compress(c, preset=9)}
    body, data, first = bytearray(), bytearray(), None
    for i in range(40):
        t = (6, 7, 5)[i % 3]
        n = int(r.choice([1024, 8192, 32768, 131072, 262144 if t == 6 else 131072]))
        c = inputs.make(kinds[i % len(kinds)], n, 500 + i)
        p = enc[t](c)
        first = first if first is not None else p
        body += MARKER + bytes([t, 0]) + struct.pack("<III", n, n, len(p)) + p
        data += c
    body += MARKER + bytes(12)
    return bytes(body), bytes(data), first


def test_container_types_5_6_7(eng):
    import torch
    body, data, first = _body(5)
    t = torch.frombuffer(bytearray(body), dtype=torch.uint8).cuda()
    known = eng.method_mask([1, 2, 3, 4, 5, 6, 7])
    for gpu_index in (True, False):
        dec, status = eng.decompress_device(t, len(data), known_mask=known, gpu_index=gpu_index)
        assert status == [0, 0] and bytes(dec.cpu().numpy()) == data
    out, status = eng.decompress_host(np.frombuffer(body, dtype=np.uint8), len(data), known_mask=known)
    assert status == [0, 0] and out.tobytes() == data
    # bits 6 and 7 cleared: those payloads are copied through (adaptive_compressor.py:432-435)
    dec, status = eng.decompress_device(t, len(data), known_mask=eng.method_mask([1, 2, 3, 4, 5]))
    assert bytes(dec.cpu().numpy())[:len(first)] == first
    # a package whose stream is broken decodes to zeros and is counted
    bad = bytearray(body)
    bad[18 + len(first) - 3] ^= 1
    tb = torch.frombuffer(bad, dtype=torch.uint8).cuda()
    dec, status = eng.decompress_device(tb, len(data), known_mask=known)
    n0 = struct.unpack("<I", body[6:10])[0]
    assert status == [1, 0] and bytes(dec.cpu().numpy()) == bytes(n0) + data[n0:]


def _ambc_file(path, body, data):
    header_body = bytes([32]) + MARKER + b"\x01" + hashlib.md5(data).digest() + struct.pack("<QQ", len(data), len(body))
    hdr = b"AMBC" + bytes([2]) + struct.pack("<I", 9 + len(header_body)) + header_body
    with open(path, "wb") as f:
        f.write(hdr + body)


def test_facade_and_cli(eng, tmp_path):
    from adaptive_compression_b200 import AdaptiveCompressor
    body, data, _ = _body(9)
    src, dst = str(tmp_path / "in.ambc"), str(tmp_path / "out.bin")
    _ambc_file(src, body, data)
    c = AdaptiveCompressor(methods=[1, 2, 3, 4, 5, 6, 7])
    c.decompress(src, dst)
    assert c.last_status == [0, 0] and open(dst, "rb").read() == data
    with pytest.raises(ValueError, match="Checksum mismatch"):
        AdaptiveCompressor().decompress(src, dst)
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "main.py"), "decompress", src, dst, "--methods",
                        "deflate,bzip2,lzma"], capture_output=True, text=True, env=env, cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout + r.stderr
    assert open(dst, "rb").read() == data
    r = subprocess.run([sys.executable, os.path.join(ROOT, "main.py"), "decompress", src, dst], capture_output=True,
                       text=True, env=env, cwd=str(tmp_path))
    assert r.returncode == 1 and "Checksum mismatch" in r.stdout
    # the plug-in objects decode on the GPU
    from adaptive_compression_b200.compression_methods import BZip2Compression, LZMACompression
    d = inputs.make("log", 70000, 12)
    assert BZip2Compression().decompress(bz2.compress(d), len(d)) == d
    assert LZMACompression().decompress(lzma.compress(d), len(d)) == d
    assert LZMACompression().decompress(lzma.compress(d), 100) == d[:100]
