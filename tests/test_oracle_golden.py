"""CPU: pin the C oracle (oracle/ambc_oracle.c) to the golden vectors produced by the
unmodified Python reference (oracle/make_golden.py)."""
import hashlib

import pytest

import inputs
import oracle as O


def sha(b):
    return hashlib.sha256(b).hexdigest()


ERR = {"IndexError": O.ERR_INDEX, "ValueError": O.ERR_VALUE}


def test_codec_kat(golden):
    cases = dict(inputs.codec_cases())
    for row in golden["codec_kat"]:
        data = cases[row["name"]]
        assert sha(data) == row["sha256"], row["name"]
        for mid_s, ent in row["methods"].items():
            mid = int(mid_s)
            assert O.should_use(mid, data) == ent["should_use"], (row["name"], mid)
            got = O.compress(mid, data)
            if "error" in ent:
                assert got == ERR[ent["error"]], (row["name"], mid)
                continue
            assert isinstance(got, bytes), (row["name"], mid, got)
            assert len(got) == ent["len"] and sha(got) == ent["sha256"], (row["name"], mid)
            if mid == 2:  # indexed search == the reference's naive scan
                assert O.compress(2, data, lz_fast=True) == got, row["name"]
            if ent["roundtrip"] is True:
                assert O.decompress(mid, got, len(data)) == data, (row["name"], mid)


def test_decode_kat(golden):
    for row in golden["decode_kat"]:
        got = O.decompress(row["method"], bytes.fromhex(row["payload"]), row["orig_len"])
        if row["error"]:
            assert got == ERR[row["error"]], row["name"]
        else:
            assert got == bytes.fromhex(row["out"]), row["name"]


def test_gates_kat(golden):
    for row in golden["gates_kat"]:
        k, n, frac, data = inputs.gate_case(row["i"])
        assert sha(data) == row["sha256"]
        assert [O.should_use(m, data) for m in (1, 2, 3, 4)] == row["gates"], row


def test_marker_kat(golden):
    cases = {c[0]: c for c in inputs.marker_cases()}
    for row in golden["marker_kat"]:
        _, data, max_len, sample = cases[row["name"]]
        assert sha(data) == row["sha256"]
        if row["marker"] is None:
            with pytest.raises(ValueError):
                O.find_marker(data, max_len, sample)
        else:
            b, L = O.find_marker(data, max_len, sample)
            assert (b.hex(), L) == (row["marker"], row["length"]), row["name"]


def _cfg(row):
    cfg = row["cfg"]
    marker = (O.FIXED_MARKER, 32)
    return cfg, marker


def test_container_kat(golden):
    cases = {c[0]: c for c in inputs.container_cases()}
    for row in golden["container_kat"]:
        name, data, _ = cases[row["name"]]
        cfg = row["cfg"]
        assert sha(data) == row["sha256"]
        marker = (O.FIXED_MARKER, 32)
        if cfg.get("found_marker"):
            marker = O.find_marker(data, 32)
        out, raw, pm = O.compress_file(data, cfg["chunk_size"], tuple(cfg.get("method_ids", (1, 2, 3, 4))), marker,
                                       bool(cfg.get("per_chunk_raw")), lz_fast=False)
        assert raw == row["stored_verbatim"], name
        assert len(out) == row["ambc_len"] and sha(out) == row["ambc_sha256"], name
        if not raw:
            assert [list(p) for p in pm] == row["packages"], name
            assert O.decompress_file(out) == data, name


def test_md5():
    for n in (0, 1, 55, 56, 63, 64, 65, 119, 120, 1000, 4096):
        d = inputs.rand(n, 900 + n)
        assert O.md5(d) == hashlib.md5(d).digest()


def test_fast_lz_equals_naive_fuzz():
    import numpy as np
    r = np.random.RandomState(7)
    kinds = sorted(inputs.KINDS)
    for i in range(60):
        k = kinds[r.randint(len(kinds))]
        n = int(r.choice([1, 2, 3, 7, 64, 500, 2048, 4096, 4097, 6000, 8192]))
        d = inputs.make(k, n, 7000 + i)
        assert O.compress(2, d, lz_fast=True) == O.compress(2, d), (k, n, i)


def test_container_dynamic_kat(golden):
    """multi-candidate (dynamic chunk size) files written by the unmodified reference
    (adaptive_compressor.py:548-584, default and custom candidate lists) == oracle, byte for byte"""
    cases = {n: (d, c) for n, d, c in inputs.dynamic_cases()}
    for row in golden["container_dyn_kat"]:
        data, cfg = cases[row["name"]]
        assert sha(data) == row["sha256"]
        f, raw, pm = O.compress_file(data, tuple(cfg["chunk_size"]), tuple(cfg.get("method_ids", (1, 2, 3, 4))))
        assert len(f) == row["ambc_len"] and sha(f) == row["ambc_sha256"], row["name"]
        assert [list(p) for p in pm] == row["packages"], row["name"]
        assert O.decompress_file(f) == data
