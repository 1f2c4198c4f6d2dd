"""GPU parity, per codec: the CUDA encoders / decoders / gates called through the C-ABI
(adaptive_compression_b200.engine -> libambc.so) against the CPU oracle and the golden vectors of the
unmodified reference.  Bit-exact."""
import hashlib

import numpy as np
import pytest

import inputs
import oracle as O

pytestmark = pytest.mark.gpu


def sha(b):
    return hashlib.sha256(b).hexdigest()


ERRN = {"IndexError": -1, "ValueError": -2}


@pytest.fixture(scope="module")
def eng():
    from adaptive_compression_b200 import engine
    engine.require_cuda()
    return engine


def _fmt(x):
    return x if isinstance(x, int) else "%d:%s" % (len(x), sha(x)[:12])


@pytest.mark.parametrize("mid", [1, 2, 3, 4])
def test_encode_golden(eng, golden, mid):
    """payload bytes == the reference's own compress() output (golden) for every KAT input"""
    cases = dict(inputs.codec_cases())
    names = [r["name"] for r in golden["codec_kat"] if r["n"] > 0]
    got = eng.codec_encode_batch(mid, [cases[n] for n in names])
    bad = []
    for row, g in zip([r for r in golden["codec_kat"] if r["n"] > 0], got):
        ent = row["methods"][str(mid)]
        if "error" in ent:
            ok = g == ERRN[ent["error"]]
        else:
            ok = isinstance(g, bytes) and len(g) == ent["len"] and sha(g) == ent["sha256"]
        if not ok:
            bad.append((row["name"], _fmt(g), ent.get("len"), ent.get("error")))
    assert not bad, bad


def test_gates_golden(eng, golden):
    rows = [r for r in golden["gates_kat"] if r["n"] > 0]
    datas = [inputs.gate_case(r["i"])[3] for r in rows]
    gates, ent = eng.should_use_batch(datas)
    bad = []
    for r, g, d, h in zip(rows, gates, datas, ent):
        if [g[m] for m in (1, 2, 3, 4)] != r["gates"]:
            bad.append((r["i"], r["kind"], r["n"], [g[m] for m in (1, 2, 3, 4)], r["gates"], h))
        if r["n"] >= 100:
            assert abs(h - O.entropy(d)) < 1e-9, (r["i"], h, O.entropy(d))
    assert not bad, bad


def test_gates_codec_cases(eng, golden):
    cases = dict(inputs.codec_cases())
    rows = [r for r in golden["codec_kat"] if r["n"] > 0]
    gates, _ = eng.should_use_batch([cases[r["name"]] for r in rows])
    bad = [(r["name"], g) for r, g in zip(rows, gates)
           if [g[m] for m in (1, 2, 3, 4)] != [r["methods"][str(m)]["should_use"] for m in (1, 2, 3, 4)]]
    assert not bad, bad


def _capacity_case(mid, n):
    """an input whose payload reaches the top of the encoders' payload capacity (2 * 8192 bytes)"""
    r = np.random.RandomState(n)
    if mid == 1:  # no two equal neighbours: one pair per byte, 2n bytes
        a = np.cumsum(r.randint(1, 256, size=n)) % 256
    elif mid == 2:  # random bytes: (almost) only literals, about 2n bytes
        a = r.randint(0, 256, size=n)
    else:  # exactly 255 values, near uniform: an 8-bit code, about 1280 + n bytes
        a = r.permutation(np.arange(n) % 255)
    return bytes(a.astype(np.uint8))


@pytest.mark.parametrize("mid", [1, 2, 3, 4])
def test_encode_fuzz_vs_oracle(eng, mid):
    """seeded inputs of every kind and many sizes, and the largest payloads: CUDA payload == oracle payload"""
    r = np.random.RandomState(100 + mid)
    kinds = sorted(inputs.KINDS)
    datas = []
    for i in range(300):
        k = kinds[r.randint(len(kinds))]
        n = int(r.choice([1, 2, 3, 4, 5, 31, 32, 33, 100, 127, 128, 129, 255, 256, 257, 511, 777, 1024, 2048,
                          3000, 4095, 4096, 4097, 5000, 8191, 8192]))
        d = inputs.make(k, n, 20000 + 1000 * mid + i)
        if r.randint(4) == 0 and n > 16:  # noise injection
            a = np.frombuffer(d, dtype=np.uint8).copy()
            m = r.rand(n) < r.choice([0.01, 0.1, 0.5])
            a[m] = r.randint(0, 256, size=int(m.sum()))
            d = a.tobytes()
        datas.append(d)
    datas += [_capacity_case(mid, n) for n in (4096, 4097, 8192)]
    got = eng.codec_encode_batch(mid, datas)
    bad = []
    for i, (d, g) in enumerate(zip(datas, got)):
        want = O.compress(mid, d, lz_fast=True)
        if g != want:
            bad.append((i, len(d), _fmt(g), _fmt(want)))
    assert not bad, bad[:20]


@pytest.mark.parametrize("mid", [1, 2, 3, 4, 255])
def test_decode_roundtrip_and_oracle(eng, mid):
    r = np.random.RandomState(200 + mid)
    kinds = sorted(inputs.KINDS)
    payloads, origs, datas = [], [], []
    for i in range(200):
        k = kinds[r.randint(len(kinds))]
        n = int(r.choice([1, 2, 3, 5, 32, 100, 129, 256, 1000, 2048, 4096, 6000, 8192]))
        d = inputs.make(k, n, 30000 + 1000 * mid + i)
        p = O.compress(mid, d, lz_fast=True)
        if isinstance(p, int):
            continue
        payloads.append(p)
        datas.append(d)
        # mostly the true length, sometimes shorter / longer (truncate / pad semantics)
        origs.append(n if r.randint(5) else max(0, n + int(r.randint(-40, 40))))
    got = eng.codec_decode_batch(mid, payloads, origs)
    bad = []
    for i, (p, o, d, g) in enumerate(zip(payloads, origs, datas, got)):
        want = O.decompress(mid, p, o)
        if g != want:
            bad.append((i, len(p), o, _fmt(g), _fmt(want)))
        if o == len(d) and want != d:
            bad.append(("oracle-roundtrip", i))
    assert not bad, bad[:20]


def test_decode_golden_malformed(eng, golden):
    """decoder edge cases incl. the reference's quirks (SURVEY.md §3.3), outputs from the reference"""
    bad = []
    for mid in (1, 2, 3, 4, 255):
        rows = [r for r in golden["decode_kat"] if r["method"] == mid]
        got = eng.codec_decode_batch(mid, [bytes.fromhex(r["payload"]) for r in rows], [r["orig_len"] for r in rows])
        for r, g in zip(rows, got):
            want = ERRN[r["error"]] if r["error"] else bytes.fromhex(r["out"])
            if g != want:
                bad.append((r["name"], _fmt(g), _fmt(want)))
    assert not bad, bad


def test_decode_corrupted_fuzz(eng):
    """random corruption of valid payloads: same bytes / same error as the oracle"""
    r = np.random.RandomState(77)
    bad = []
    for mid in (1, 2, 3, 4):
        payloads, origs = [], []
        for i in range(150):
            d = inputs.make(sorted(inputs.KINDS)[r.randint(len(inputs.KINDS))], int(r.choice([64, 300, 1024, 4096])), 40000 + i)
            p = O.compress(mid, d, lz_fast=True)
            if isinstance(p, int):
                continue
            payloads.append(inputs.corrupt(p, r))
            origs.append(len(d))
        got = eng.codec_decode_batch(mid, payloads, origs)
        for i, (p, o, g) in enumerate(zip(payloads, origs, got)):
            want = O.decompress(mid, p, o)
            if g != want:
                bad.append((mid, i, len(p), o, _fmt(g), _fmt(want)))
    assert not bad, bad[:20]


def test_encode_dictionary_seeded_sizes(eng):
    """Dictionary items of 3, 100, 1000 and 4096 bytes of every kind: same payloads as the oracle"""
    r = np.random.RandomState(555)
    kinds = sorted(inputs.KINDS)
    datas = [inputs.make(kinds[r.randint(len(kinds))], int(r.choice([3, 100, 1000, 4096])), 50000 + i) for i in range(60)]
    got = eng.codec_encode_batch(2, datas)
    bad = [(i, len(d)) for i, (d, g) in enumerate(zip(datas, got)) if g != O.compress(2, d, lz_fast=True)]
    assert not bad, bad


def test_huffman_decode_code_shapes(eng):
    """the code shapes that steer k_decode_warp's Huffman paths (decode_warp.cuh): flat codes (ranges must be a
    multiple of the code length), near-flat codes that never re-synchronise (all-entries path), codes longer
    than the look-up table (tree walk), streams shorter than a lane's range, orig_len below / above the number
    of symbols in the stream -- every output equals the oracle's decoder (compression_methods.py:407-470)"""
    r = np.random.RandomState(4242)
    datas = []
    for k in (2, 3, 4, 5, 7, 8, 9, 12, 16, 17, 32, 33, 64, 100, 128, 200, 255):  # (near-)uniform alphabets
        for n in (100, 517, 4096, 8192):
            datas.append(bytes(r.randint(0, k, size=n).astype(np.uint8)))
    for n in (300, 4096, 8192):  # exactly equal counts: flat trees
        for k in (2, 4, 8, 16, 64):
            datas.append(bytes(np.tile(np.arange(k, dtype=np.uint8), n // k + 1)[:n]))
    for n in (2000, 4096, 8192):  # geometric and Fibonacci-like counts: codes of 12 .. 20 bits
        sym, cnt, out = 0, n // 2, []
        while cnt >= 1 and sym < 40:
            out += [sym] * int(cnt); sym += 1; cnt = cnt * 0.62
        a = np.array(out[:n], dtype=np.uint8); r.shuffle(a)
        datas.append(bytes(a))
        datas.append(inputs.make("fib", n, 77 + n))
    payloads, origs = [], []
    for d in datas:
        p = O.compress(3, d)
        if isinstance(p, int):
            continue
        for o in (len(d), max(0, len(d) - 37), len(d) + 19, 1):
            payloads.append(p); origs.append(o)
    got = eng.codec_decode_batch(3, payloads, origs)
    bad = [(i, len(p), o, _fmt(g)) for i, (p, o, g) in enumerate(zip(payloads, origs, got)) if g != O.decompress(3, p, o)]
    assert not bad, bad[:20]
    # the same payloads framed as packages of a body: the container path of the same kernel
    body = bytearray()
    want = bytearray()
    for p, o in zip(payloads, origs):
        w = O.decompress(3, p, o)
        if o == 0 or len(p) > 8192 or not isinstance(w, bytes) or len(w) != o:
            continue
        body += b"\xff\xff\x00\x00" + bytes([3, 0]) + int(o).to_bytes(4, "little") * 2 + len(p).to_bytes(4, "little") + p
        want += w
    body += b"\xff\xff\x00\x00" + bytes(12)
    import torch
    dec, status = eng.decompress_device(torch.frombuffer(bytearray(body), dtype=torch.uint8).cuda(), len(want))
    assert status == [0, 0] and bytes(dec.cpu().numpy()) == bytes(want)
