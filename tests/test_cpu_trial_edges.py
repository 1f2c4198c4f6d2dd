"""The boundary cases of tests/trial_edges.py sit where their labels say, on the oracle, without a GPU.

Every case's numbers are recomputed from scratch and checked against its label and side; the integer predicates
sf_select uses in place of the reference's fp64 quotients agree with the oracle's gates on every case; the ledger
holds every (label, side) of WANT in each k_select_fast instantiation; and every case's outcome is the one
O.compress_body chooses."""
import time

import numpy as np
import pytest

import oracle as O
import trial_edges as T

_ALL = (-1, 0, 1)
# label -> {instantiation (4096: chunks of <= 4096 bytes, 8192: 4097..8192) -> sides that must be present}
WANT = {
    "rle_gate": {4096: {-10, 0, 10, -7, 3, -3, 7, -6, 4}, 8192: {-7, 3}},
    "dict_gate": {4096: {-10, 0, 10, -4, 6, -2, 8}, 8192: {-10, 0, 10}},
    "huff_K": {4096: {1, 2, 255, 256}, 8192: {1, 2, 255, 256}},
    "huff_n": {4096: {99, 100}},
    "huff_H7": {4096: {0}, 8192: {0}},
    "huff_near7": {4096: {-2, -1, 1, 2}, 8192: {-2, -1, 1, 2}},
    "dict_huff": {4096: set(_ALL), 8192: set(_ALL)},
    "rle_huff": {4096: set(_ALL)},
    "rle_dict": {4096: {-2, 0, 2}},
    "rle_eq_lzmin": {4096: {-2, 0, 2}},
    "rle_eq_hfmin": {4096: {-2, 0, 2}},
    "benefit_rle": {4096: set(_ALL)},
    "benefit_huff": {4096: set(_ALL), 8192: set(_ALL)},
    "benefit_dict": {4096: set(_ALL), 8192: set(_ALL)},
    "staged": {4096: {(339, 0), (339, 1), (340, 0), (340, 1)}},
    "hopeless": {4096: set(_ALL), 8192: set(_ALL)},
    "hopeless_exact": {4096: set(_ALL), 8192: set(_ALL)},
    "size": {4096: {31, 32, 99, 100, 127, 128, 129, 4096}, 8192: {4097, 8191, 8192}},
    "short_last": {4096: {1, 3, 31, 32, 99, 100, 127, 128}, 8192: {1, 3, 31, 32, 99, 100, 127, 128}},
    "methods": {k: {(1,), (2,), (3,), (2, 3), (1, 3), (1, 2, 3)} for k in (4096, 8192)},
    "window": {8192: {4095, 4096, 4097}},
    "match_len": {4096: {31, 32, 33, 34}},
    "match_to_end": {k: {33, 32, 31, 4, 3} for k in (4096, 8192)},
    "match_at_n-3": {k: {0, 77} for k in (4096, 8192)},
    "three_byte_subbuckets": {4096: {4096}, 8192: {8192}},
    "overlap": {k: {1, 2, 3} for k in (4096, 8192)},
    "big_bucket": {4096: {455}, 8192: {910}},
    "no_merge": {k: {37} for k in (4096, 8192)},
    "ratio_tie": {4096: set(_ALL)},
}
BENEFIT = ("benefit_rle", "benefit_huff", "benefit_dict")
MATCH = ("window", "match_len", "match_to_end", "match_at_n-3", "three_byte_subbuckets", "overlap", "big_bucket",
         "no_merge")


def case_inst(c):
    """the instantiation the fixed grid (or, for candidate lists, the span encoder of the largest size) runs"""
    return T.inst(c.chunk if isinstance(c.chunk, int) else max(c.chunk))


_T0 = time.time()
_CASES = T.cases()
BUILD_SECONDS = time.time() - _T0


def test_construction_time():
    print("trial_edges: %d cases built in %.1f s" % (len(_CASES), BUILD_SECONDS))
    assert BUILD_SECONDS < 60


def _check_side(c, m):
    """assert that numbers m of case c put it where (label, side) says"""
    L, s, n, p, g = c.label, c.side, m["n"], m["pay"], m["gate"]
    if L == "rle_gate":
        assert s == 10 * m["rep"] - 3 * (m["ss"] - 1)
    elif L == "dict_gate":
        assert s == 10 * m["distinct3"] - 8 * m["ss"]
    elif L == "huff_K":
        assert m["K"] == s and m["H"] < 7.0 and g[3]
        assert (p[3] is not None) == (2 <= s <= 255)  # the encoder rejects one symbol and 256 symbols
    elif L == "huff_n":
        assert n == s and m["H"] < 7.0
    elif L == "huff_H7":
        assert m["H"] == 7.0 and not g[3]
    elif L == "huff_near7":
        d = m["H"] - 7.0
        assert np.sign(d) == np.sign(s) and (0 < abs(d) < 0.02 if abs(s) == 1 else 0.02 < abs(d) < 0.03), d
    elif L == "dict_huff":
        assert g[2] and g[3] and p[2] - p[3] == s and not g[1]
        assert m["chosen"] == ((2, p[2]) if s <= 0 else (3, p[3]))
    elif L == "rle_huff":
        assert g[1] and g[3] and p[1] - p[3] == s
        assert m["chosen"] == ((1, p[1]) if s <= 0 else (3, p[3]))
        assert p[1] > T.hf_min(n)  # the Huffman payload is built and compared, no outright RLE win
    elif L == "rle_dict":
        assert g[1] and g[2] and p[1] - p[2] == s
        assert m["chosen"][0] == (1 if s <= 0 else 2) or 3 in c.methods
    elif L == "rle_eq_lzmin":
        assert g[1] and p[1] - T.lz_min(n) == s and m["chosen"] == (1, p[1])
    elif L == "rle_eq_hfmin":
        assert g[1] and p[1] - T.hf_min(n) == s
        assert m["chosen"] == ((1, p[1]) if p[1] <= p[3] else (3, p[3]))
    elif L in BENEFIT:
        mid = {"benefit_rle": 1, "benefit_huff": 3, "benefit_dict": 2}[L]
        live = [k for k in (1, 2, 3) if T.RANGE[k][0] <= n <= T.RANGE[k][1] and g[k] and p[k] is not None]
        assert live == [mid], live  # the only method with a payload (Huffman fails on K = 256)
        assert p[mid] + m["ovh"] - n == s
        assert m["chosen"] == ((mid, p[mid]) if s < 0 else (255, n))
    elif L == "staged":
        per, tgt = s
        assert m["distinct3"] == per and 100 * per - 34 * m["ss"] in (-100, 0)
        assert g[2] and g[3] and p[2] - p[3] == tgt
        rest, lb = T.staged_checks(O.compress(2, c.data, lz_fast=True), n)[1]
        assert rest % 32 == 0 and lb == p[2]  # the abort bound is tight at the second stage boundary
        assert m["chosen"] == ((2, p[2]) if tgt == 0 else (3, p[3]))
    elif L in ("hopeless", "hopeless_exact"):
        a = np.frombuffer(c.data, dtype=np.uint8)
        hashed, exact = T.ngram_bound(a, hashed=True), T.ngram_bound(a)
        assert g[2] and g[3] and not g[1] and 100 * m["distinct3"] >= 34 * m["ss"]  # `staged`: the bound is consulted
        assert p[3] + m["ovh"] < n  # cutoff = Huffman payload + 1
        assert (hashed if L == "hopeless" else exact) - (p[3] + 1) == s
        assert hashed <= exact <= p[2]  # the kernel's hash sets only lose; the bound is a lower bound
        assert m["chosen"] == (3, p[3])
    elif L == "size":
        assert n == s
    elif L == "short_last":
        assert n == s < c.chunk
    elif L == "methods":
        assert tuple(c.methods) == s
    elif L in MATCH:
        assert tuple(c.methods) == (2,) and m["chosen"] == (2, p[2])  # a beneficial Dictionary payload: bytes compared


@pytest.mark.parametrize("label", sorted(WANT))
def test_cases_sit_where_their_labels_say(label):
    got = [(c, m) for c, m in _CASES if c.label == label]
    assert got
    for c, m in got:
        if m is None:
            continue
        fresh = T.numbers(c.data, c.methods, c.marker)
        assert fresh == m, (label, c.side)
        _check_side(c, m)


def test_integer_gates_agree_with_the_oracle():
    """sf_select's integer restatements of the fp64 quotients (rep / (ss - 1) > 0.3, distinct / s < 0.8) give the
    oracle's gate on every case"""
    for c, m in _CASES:
        if m is None:
            continue
        n = m["n"]
        assert m["gate"][1] == (n >= 4 and 10 * m["rep"] > 3 * (m["ss"] - 1)), (c.label, c.side)
        assert m["gate"][2] == (n >= 100 and 10 * m["distinct3"] < 8 * m["ss"]), (c.label, c.side)
        assert m["gate"][3] == (n >= 100 and m["H"] < 7.0), (c.label, c.side)


def test_ledger_holds_every_wanted_side():
    have = {}
    for c, _ in _CASES:
        have.setdefault(c.label, {}).setdefault(case_inst(c), set()).add(c.side)
    missing = [(L, k, sorted(want - have.get(L, {}).get(k, set()), key=str))
               for L, per in WANT.items() for k, want in per.items() if not want <= have.get(L, {}).get(k, set())]
    assert not missing, missing
    # the benefit test at every package overhead (markers of 1..4 bytes: 15..18), on both sides
    for L in BENEFIT:
        for k in WANT[L]:
            got = {(len(c.marker), c.side) for c, _ in _CASES if c.label == L and case_inst(c) == k}
            assert got >= {(mb, s) for mb in (1, 2, 3, 4) for s in _ALL}, (L, k)
    # ratio ties under both candidate lists
    assert {c.chunk for c, _ in _CASES if c.label == "ratio_tie"} == {(4096, 2048, 1024), (3072, 1536, 512)}


def test_outcomes_match_compress_body():
    """every single-chunk case: the oracle's body writer picks the chosen (type, len) of its numbers"""
    for c, m in _CASES:
        if m is None:
            continue
        _, pm = O.compress_body(c.data, c.chunk, c.methods, c.marker, per_chunk_raw=True)
        assert [tuple(x) for x in pm] == [(m["chosen"][0], m["n"], m["chosen"][1])], (c.label, c.side)


def test_ratio_ties_pick_as_labelled():
    """(len + ovh) / size equal for the two largest candidates (side 0) and one RLE run either side: the larger
    candidate keeps the tie"""
    for c, _ in _CASES:
        if c.label != "ratio_tie":
            continue
        big, half, small = c.chunk
        a = c.data
        ovh = len(c.marker) + 14
        p1, p2, p3 = (len(O.compress(1, a[:k])) for k in (big, half, small))
        for k, pk in ((big, p1), (half, p2)):  # RLE is the winner of both tied candidates
            assert O.compress_body(a[:k], k, c.methods, c.marker)[1] == [(1, k, pk)]
        assert (p1 + ovh) - 2 * (p2 + ovh) == 2 * c.side
        assert (p3 + ovh) * half > (p2 + ovh) * small
        _, pm = O.compress_body(a, c.chunk, c.methods, c.marker)
        assert pm[0][1] == (big if c.side <= 0 else half), c.side
