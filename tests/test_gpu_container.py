"""GPU parity, whole body: the CUDA select / scan / pack path and the decode path through the
C-ABI against the oracle and the golden .ambc files of the unmodified reference."""
import hashlib

import numpy as np
import pytest

import inputs
import oracle as O

pytestmark = pytest.mark.gpu


def sha(b):
    return hashlib.sha256(b).hexdigest()


@pytest.fixture(scope="module")
def eng():
    from adaptive_compression_b200 import engine
    engine.require_cuda()
    return engine


def gpu_body(eng, data, chunk, methods=(1, 2, 3, 4), marker=O.FIXED_MARKER, pcr=False):
    t = eng.to_device(data)
    o = eng.compress_device(t, chunk, eng.method_mask(methods), 1 if pcr else 0, marker)
    return o.body.cpu().numpy().tobytes(), eng.package_map(o, len(data), chunk, pcr), o


def test_body_matches_golden_reference_files(eng, golden):
    """body bytes == bytes 47.. of the .ambc the unmodified reference wrote"""
    cases = {c[0]: c for c in inputs.container_cases()}
    bad = []
    for row in golden["container_kat"]:
        name, data, _ = cases[row["name"]]
        cfg = row["cfg"]
        if not data:
            continue
        marker = O.FIXED_MARKER
        if cfg.get("found_marker"):
            mb, ml = O.find_marker(data, 32)
            marker = O.marker_aligned(mb, ml)
        want_file, raw, want_pm = O.compress_file(data, cfg["chunk_size"], tuple(cfg.get("method_ids", (1, 2, 3, 4))),
                                                  (O.FIXED_MARKER, 32) if not cfg.get("found_marker") else O.find_marker(data, 32),
                                                  bool(cfg.get("per_chunk_raw")))
        body, pm, o = gpu_body(eng, data, cfg["chunk_size"], tuple(cfg.get("method_ids", (1, 2, 3, 4))), marker,
                               bool(cfg.get("per_chunk_raw")))
        wbody, wpm = O.compress_body(data, cfg["chunk_size"], tuple(cfg.get("method_ids", (1, 2, 3, 4))), marker,
                                     bool(cfg.get("per_chunk_raw")))
        if body != wbody or [tuple(p) for p in pm] != [tuple(p) for p in wpm]:
            bad.append((name, len(body), len(wbody), pm[:6], wpm[:6]))
            continue
        if not row["stored_verbatim"]:
            hs = 43 + len(marker)
            assert sha(want_file) == row["ambc_sha256"]
            assert want_file[hs:] == body, name
            assert [list(p) for p in pm] == row["packages"], name
    assert not bad, bad


@pytest.mark.parametrize("chunk", [512, 1024, 2048, 4096, 8192, 3000])
def test_body_fuzz_vs_oracle(eng, chunk):
    r = np.random.RandomState(chunk)
    bad = []
    for it in range(6):
        nch = int(r.randint(3, 40))
        data = inputs.mixed_file(nch, chunk, 5000 + chunk + it) + inputs.text(int(r.randint(0, chunk)), it)
        pcr = bool(it % 2)
        if it == 3:  # a random chunk in the middle: tail-raw rule / per-chunk raw
            data = data[:chunk * 2] + inputs.rand(chunk, it) + data[chunk * 2:]
        body, pm, o = gpu_body(eng, data, chunk, pcr=pcr)
        wbody, wpm = O.compress_body(data, chunk, per_chunk_raw=pcr)
        if body != wbody:
            first = next((i for i, (a, b) in enumerate(zip(body, wbody)) if a != b), min(len(body), len(wbody)))
            bad.append((chunk, it, len(body), len(wbody), first, pm[:8], wpm[:8]))
            continue
        out, status = eng.decompress_device(o.body, len(data), body_host=np.frombuffer(body, dtype=np.uint8))
        if out.cpu().numpy().tobytes() != data or status != [0, 0]:
            bad.append(("roundtrip", chunk, it, status))
    assert not bad, bad


def test_selection_small_alphabets_vs_oracle(eng):
    """the Huffman-first order of k_select_fast and its early stop of a Dictionary trial that cannot win
    (small alphabets, varying skew, sprinkled repeats and runs) never change the outcome: body and
    method map equal to the oracle's in-order trial of every method (adaptive_compressor.py:537-590)"""
    r = np.random.RandomState(77)
    seen = np.zeros(5, dtype=np.int64)
    for it in range(60):
        chunk = int(r.choice([1024, 2048, 4096, 4096, 3000]))
        parts = []
        for _ in range(int(r.randint(3, 16))):
            n = chunk if r.rand() < 0.8 else int(r.randint(1, chunk + 1))
            K = int(r.choice([2, 3, 4, 6, 8, 12, 16, 20, 32, 64, 128, 200]))
            w = r.rand(K) ** float(r.choice([0.5, 1, 2, 4, 8]))
            a = r.choice(K, size=n, p=w / w.sum()).astype(np.uint8)
            a = (a * int(r.choice([1, 3, 7])) + int(r.randint(0, 200))).astype(np.uint8)
            for _ in range(int(r.choice([0, 2, 30, 100, 300, 600]))):
                L = int(r.choice([3, 4, 5, 7, 8, 9, 12, 16, 31, 32, 40]))
                if n > 2 * L + 2:
                    s_, d_ = int(r.randint(0, n - L)), int(r.randint(0, n - L))
                    a[d_:d_ + L] = a[s_:s_ + L].copy()
            if r.rand() < 0.15:
                s_ = int(r.randint(0, n)); a[s_:s_ + int(r.randint(1, 600))] = int(r.randint(256))
            parts.append(a)
        data = np.concatenate(parts).tobytes()
        body, pm, o = gpu_body(eng, data, chunk)
        want, wpm = O.compress_body(data, chunk)
        assert [tuple(p) for p in pm] == [tuple(p) for p in wpm], (it, chunk)
        assert body == want, (it, chunk)
        seen += np.array(o.usage[:5])
    assert seen[1] and seen[2] and seen[3], seen  # RLE, Dictionary and Huffman winners all occur


def test_method_masks(eng):
    data = inputs.mixed_file(10, 4096, 909)
    for methods in [(1,), (2,), (3,), (4,), (1, 3), (2, 4), (1, 2, 3, 4), ()]:
        body, pm, o = gpu_body(eng, data, 4096, methods)
        wbody, wpm = O.compress_body(data, 4096, methods)
        assert body == wbody, methods
        assert [tuple(p) for p in pm] == [tuple(p) for p in wpm], methods


def test_decode_reference_files(eng, golden):
    """the CUDA decoder reads what the reference wrote (via the oracle restatement, pinned by sha256)"""
    cases = {c[0]: c for c in inputs.container_cases()}
    for row in golden["container_kat"]:
        name, data, _ = cases[row["name"]]
        cfg = row["cfg"]
        if row["stored_verbatim"] or not data:
            continue
        marker = (O.FIXED_MARKER, 32) if not cfg.get("found_marker") else O.find_marker(data, 32)
        f, raw, _ = O.compress_file(data, cfg["chunk_size"], tuple(cfg.get("method_ids", (1, 2, 3, 4))), marker,
                                    bool(cfg.get("per_chunk_raw")))
        assert sha(f) == row["ambc_sha256"]
        hs = int.from_bytes(f[5:9], "little")
        body = np.frombuffer(f[hs:], dtype=np.uint8)
        out, status = eng.decompress_device(eng.to_device(body), len(data), O.marker_aligned(*marker), body_host=body)
        assert out.cpu().numpy().tobytes() == data, name
        assert status == [0, 0], name


def test_synthetic_corpus_roundtrip_and_oracle(eng):
    """device-generated corpus (the bench workload): body == oracle on 2 MiB, round trip on 64 MiB"""
    n = 2 << 20
    t = eng.synth(n, offset=0)
    data = t.cpu().numpy().tobytes()
    o = eng.compress_device(t, 4096)
    body = o.body.cpu().numpy().tobytes()
    wbody, wpm = O.compress_body(data, 4096)
    assert body == wbody
    assert [tuple(p) for p in eng.package_map(o, n, 4096)] == [tuple(p) for p in wpm]
    n = 64 << 20
    t = eng.synth(n, offset=123 * 65536)
    o = eng.compress_device(t, 4096)
    out, status = eng.decompress_device(o.body, n)
    assert status == [0, 0]
    import torch
    assert torch.equal(out, t)
    assert o.first_raw == -1, "bench corpus must have a native winner in every chunk"


@pytest.mark.parametrize("chunk", [1024, 4096, 16384])
def test_config3_chunk_sweep_log_corpus(eng, chunk):
    """BASELINE configs[2]: chunk-size sweep on a log corpus.  1024 / 4096 against the oracle;
    16384 is degenerate under reference semantics (no native method is eligible above 8192,
    adaptive_compressor.py:114-127): the body is one raw package"""
    import torch
    n = 4 << 20
    t = eng.synth(n, offset=0, kind_mask=1 << 1)  # log kind only
    data = t.cpu().numpy().tobytes()
    o = eng.compress_device(t, chunk)
    body = o.body.cpu().numpy().tobytes()
    wbody, wpm = O.compress_body(data, chunk)
    assert body == wbody
    assert [tuple(p) for p in eng.package_map(o, n, chunk)] == [tuple(p) for p in wpm]
    if chunk == 16384:
        assert o.first_raw == 0 and len(wpm) == 1 and wpm[0][0] == 255 and len(body) == n + 18 + 16
    out, status = eng.decompress_device(o.body, n)
    assert status == [0, 0] and torch.equal(out, t)


@pytest.mark.parametrize("pcr", [False, True])
def test_config5_interleaved_segments(eng, pcr):
    """BASELINE configs[4]: high-entropy / run-heavy / low-cardinality segments interleaved at 4 KiB.
    Strict semantics send everything after the first chunk without a winner to one raw package
    (adaptive_compressor.py:586-590); the labelled per-chunk-raw extension switches method per chunk"""
    import torch
    from adaptive_compression_b200 import _lib as L
    parts = []
    for i in range(96):
        kind = ("runs", "lowcard", "rand")[i % 3] if i >= 6 else ("runs", "lowcard")[i % 2]
        parts.append(inputs.make(kind, 4096, 900 + i))
    data = b"".join(parts)
    t = eng.to_device(data)
    o = eng.compress_device(t, 4096, flags=L.F_PER_CHUNK_RAW if pcr else 0)
    body = o.body.cpu().numpy().tobytes()
    wbody, wpm = O.compress_body(data, 4096, per_chunk_raw=pcr)
    assert body == wbody
    assert [tuple(p) for p in eng.package_map(o, len(data), 4096, per_chunk_raw=pcr)] == [tuple(p) for p in wpm]
    if pcr:
        assert {p[0] for p in wpm} >= {1, 3, 255}
    else:
        assert o.first_raw == 8 and wpm[-1][0] == 255 and wpm[-1][1] == len(data) - 8 * 4096
    out, status = eng.decompress_device(o.body, len(data))
    assert status == [0, 0] and out.cpu().numpy().tobytes() == data


def test_dynamic_candidates_golden_and_oracle(eng, golden):
    """the reference's multi-candidate mode (adaptive_compressor.py:548-584): body and package list ==
    the files the unmodified reference wrote (golden) and the oracle; round trip through the decoder"""
    from adaptive_compression_b200.adaptive_compressor import AdaptiveCompressor
    cases = {n: (d, c) for n, d, c in inputs.dynamic_cases()}
    for row in golden["container_dyn_kat"]:
        data, cfg = cases[row["name"]]
        mids = tuple(cfg.get("method_ids", (1, 2, 3, 4)))
        o = eng.compress_dynamic_device(eng.to_device(data), cfg["chunk_size"], mask=eng.method_mask(mids))
        body = o.body.cpu().numpy().tobytes()
        wbody, wpm = O.compress_body(data, tuple(cfg["chunk_size"]), mids)
        assert body == wbody, row["name"]
        assert [list(p) for p in o.packages] == [list(p) for p in wpm] == row["packages"], row["name"]
        # whole file == the reference's own file
        f, raw, _ = O.compress_file(data, tuple(cfg["chunk_size"]), mids)
        assert sha(f) == row["ambc_sha256"]
        hs = int.from_bytes(f[5:9], "little")
        assert f[hs:] == body
        out, status = eng.decompress_device(o.body, len(data))
        assert status == [0, 0] and out.cpu().numpy().tobytes() == data, row["name"]


@pytest.mark.parametrize("cands", [(131072, 65536, 32768, 16384, 8192, 4096, 2048, 1024), (4096, 1024), (8192, 2048, 512)])
def test_dynamic_candidates_fuzz_vs_oracle(eng, cands):
    r = np.random.RandomState(sum(cands) % 1000)
    for i in range(7):
        kinds = ("text", "csv", "log", "runs", "lowcard", "binrec", "periodic", "rand")
        parts = [inputs.make(kinds[r.randint(len(kinds) - (0 if i % 3 == 2 else 1))], int(r.choice([700, 1024, 2048, 3000, 4096, 9000])), 6000 + 100 * i + j)
                 for j in range(int(r.randint(3, 9)))]
        data = b"".join(parts)
        # the last input allows no method at all: strict mode sends the whole file to one raw package, per-chunk-raw
        # mode cuts it into raw pieces of the smallest candidate size
        methods = () if i == 6 else (1, 2, 3, 4)
        for pcr in (False, True):
            from adaptive_compression_b200 import _lib as L
            o = eng.compress_dynamic_device(eng.to_device(data), cands, mask=eng.method_mask(methods),
                                            flags=L.F_PER_CHUNK_RAW if pcr else 0)
            wbody, wpm = O.compress_body(data, cands, methods, per_chunk_raw=pcr)
            assert o.body.cpu().numpy().tobytes() == wbody, (cands, i, pcr)
            assert [list(p) for p in o.packages] == [list(p) for p in wpm]
            if i == 6:
                assert {p[0] for p in wpm} == {255} and len(wpm) == (-(-len(data) // cands[-1]) if pcr else 1)
            out, status = eng.decompress_device(o.body, len(data))
            assert status == [0, 0] and out.cpu().numpy().tobytes() == data
