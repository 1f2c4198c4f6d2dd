"""A model of the multi-candidate ("dynamic") mode's chain walk and stitch, in plain Python over the CPU oracle.

ambc_compress_dynamic_dev (csrc/compress.cu) cuts the file into segments of 64 * g bytes, g the gcd of the candidate
sizes.  k_dynamic_walk walks a speculative chain in every segment from its first byte; the host then follows the true
chain through the segments, re-launches the walk for every (segment, entry) pair whose entry differs from the
segment's first byte (each re-entered chain stops where it meets the segment's speculative chain), repeats until no
pair is left, and assembles the chain from speculative and re-entered records.  `model()` restates that bookkeeping
step by step, so that the GPU tests can hold the library to the rounds and branches it took, not only to its body.

The winner at a position p depends only on data[p:] and on the remaining length, and the remaining length matters
only up to 8193 (candidates above 8192 bytes are eligible only when clamped to the rest of the file).  So the chain
from p up to a stop point s is the package list of the oracle's compress_body(data[p:min(n, s + 8193)]), shifted by
p: the oracle applies the reference's clamping, tie and raw rules, and the model restates none of them."""
import math

import numpy as np
import pytest

import inputs
import oracle as O

SEGU = 64           # DYN_SEGU: positions (multiples of g) per segment
HORIZON = 8193      # remaining lengths above this all give the same winner


class Chain:
    """one walk: records [(pos, size, type, comp)], exit (first position not walked), stop (strict no-winner
    position, or None), merged (a re-entered walk met the speculative chain at `exit`)"""
    __slots__ = ("entry", "recs", "exit", "stop", "merged")

    def __init__(self, entry, recs, exit, stop, merged):
        self.entry, self.recs, self.exit, self.stop, self.merged = entry, recs, exit, stop, merged


class Model:
    """spec[sg]: the speculative chain of segment sg; rounds: the (segment, entry) list of every re-launch;
    reentries: every re-entered chain, in launch order, as (round, segment, Chain); chain: the assembled
    records; entries: the (segment, entry) pairs the assembly went through; raw_from: start of the rest-of-file raw
    package (n if none)"""
    __slots__ = ("n", "g", "cmin", "seglen", "n_seg", "pcr", "spec", "rounds", "reentries", "fix", "entries", "chain",
                 "raw_from")

    @property
    def packages(self):
        """the chain as the oracle lists packages: [(type, orig, comp)]"""
        out = [(t, size, comp) for _, size, t, comp in self.chain]
        if self.raw_from < self.n:
            out.append((255, self.n - self.raw_from, self.n - self.raw_from))
        return out

    def walk_launches(self):
        """k_dynamic_walk launches: the speculative one and one per round"""
        return (1 + len(self.rounds)) if self.n else 0

    def true_positions(self):
        return {r[0] for r in self.chain} | ({self.raw_from} if self.raw_from < self.n else set())


def _walk(data, cands, methods, marker, pcr, start, end, visited=()):
    n = len(data)
    _, pm = O.compress_body(data[start:min(n, end + HORIZON)], cands, methods, marker, pcr)
    recs, pos, stop, merged = [], start, None, False
    for t, size, comp in pm:
        if pos >= end:
            break
        if pos in visited:
            merged = True
            break
        if t == 255 and not pcr:
            stop = pos  # no winner: the rest of the file is one raw package
            break
        recs.append((pos, size, t, comp))
        pos += size
    return Chain(start, recs, pos, stop, merged)


def gcd_of(cands):
    g = 0
    for c in cands:
        g = math.gcd(g, int(c))
    return g


def model(data, cands, methods=(1, 2, 3, 4), marker=O.FIXED_MARKER, pcr=False):
    """restates compress.cu's ambc_compress_dynamic_dev for a file with at least one native method"""
    data = bytes(data)
    cands = tuple(sorted({int(c) for c in cands}, reverse=True))
    n, g = len(data), gcd_of(cands)
    M = Model()
    M.n, M.g, M.cmin, M.pcr = n, g, cands[-1], pcr
    M.seglen = SEGU * g
    n_pos = -(-n // g)
    M.n_seg = -(-n_pos // SEGU)
    walk = lambda s, e, vis=(): _walk(data, cands, methods, marker, pcr, s, e, vis)  # noqa: E731
    bounds = [(sg * M.seglen, min(n, (sg + 1) * M.seglen)) for sg in range(M.n_seg)]
    M.spec = [walk(s0, s1) for s0, s1 in bounds]
    M.fix = {}  # segment -> the latest re-entered Chain (the library's fixseg / fix_entry)
    M.rounds, M.reentries = [], []
    while True:
        lst, e = [], 0
        for sg, (s0, s1) in enumerate(bounds):
            if e >= n:
                break
            if e >= s1:
                continue
            sp = M.spec[sg]
            if e == s0:
                if sp.stop is not None:
                    break
                e = sp.exit
                continue
            f = M.fix.get(sg)
            if f is not None and f.entry == e:
                last = sp if f.merged else f
                if last.stop is not None:
                    break
                e = last.exit
                continue
            lst.append((sg, e))
            if sp.stop is not None:
                break
            e = sp.exit
        if not lst:
            break
        # the library gives up past n_seg + 2 rounds; the model may not need more than that
        assert len(M.rounds) <= M.n_seg + 2, "the stitch does not settle"
        M.rounds.append(lst)
        for sg, e in lst:
            f = walk(e, bounds[sg][1], {r[0] for r in M.spec[sg].recs})
            M.fix[sg] = f
            M.reentries.append((len(M.rounds) - 1, sg, f))
    chain, raw_from, e, M.entries = [], n, 0, []
    for sg, (s0, s1) in enumerate(bounds):
        if e >= n:
            break
        if e >= s1:
            continue
        M.entries.append((sg, e))
        sp, frm = M.spec[sg], 0
        if e != s0:
            f = M.fix[sg]
            assert f.entry == e
            chain += f.recs
            if f.merged:
                frm = [r[0] for r in sp.recs].index(f.exit)  # "meeting point not on the speculative chain" if absent
            else:
                if f.stop is not None:
                    raw_from = f.stop
                    break
                e = f.exit
                continue
        chain += sp.recs[frm:]
        if sp.stop is not None:
            raw_from = sp.stop
            break
        e = sp.exit
    M.chain, M.raw_from = chain, raw_from
    return M


# ---- inputs large enough to reach the stitch ---------------------------------------------------------------------
def cascade(n, seed=501, lead=1024):
    """`lead` bytes of runs, then homogeneous text: one short package moves the true chain off the 8192 grid, and no
    segment's speculative chain meets it again, so every round resolves one more segment"""
    return inputs.runs(lead, seed) + inputs.text(n - lead, seed + 1)


def mixed(n, seed, kinds=("text", "csv", "log", "runs", "lowcard")):
    """pieces of 1..12 KiB of the given kinds"""
    r = np.random.RandomState(seed)
    parts, size = [], 0
    while size < n:
        k = kinds[r.randint(len(kinds))]
        m = int(r.randint(1, 13)) * 1024 + int(r.choice([0, 0, 256, 512, 777]))
        parts.append(inputs.make(k, m, seed * 1000 + len(parts)))
        size += m
    return b"".join(parts)[:n]


def with_noise(data, spots, seed):
    """overwrite [pos, pos + length) with random bytes for every (pos, length) in spots"""
    a = bytearray(data)
    r = np.random.RandomState(seed)
    for p, m in spots:
        a[p:p + m] = r.randint(0, 256, size=len(a[p:p + m])).astype(np.uint8).tobytes()
    return bytes(a)


REF = inputs.REF_DEFAULT_CANDIDATES
SMALL = (8192, 2048, 512)


def large_cases():
    """(name, data, cands, methods, marker, pcr): the inputs whose models the GPU tests assert coverage on"""
    out = []
    out.append(("cascade_ref_4M", cascade(4 << 20), REF, (1, 2, 3, 4), O.FIXED_MARKER, False))
    out.append(("cascade_small_3M", cascade(3 << 20, 511, 512), SMALL, (1, 2, 3, 4), O.FIXED_MARKER, False))
    out.append(("mixed_ref_2M", mixed(2 << 20, 521), REF, (1, 2, 3, 4), O.FIXED_MARKER, False))
    out.append(("mixed_small_1M", mixed(1 << 20, 522), SMALL, (1, 2, 3, 4), O.FIXED_MARKER, False))
    # random stretches that end the strict chain inside a re-entered segment or cut pcr raw pieces into it
    noisy = with_noise(mixed(1 << 20, 523), [(200_000 + 3000, 9000), (700_000, 5000)], 524)
    out.append(("noisy_small_strict", noisy, SMALL, (1, 2, 3, 4), O.FIXED_MARKER, False))
    out.append(("noisy_small_pcr", noisy, SMALL, (1, 2, 3, 4), O.FIXED_MARKER, True))
    out.append(("mixed_g256_pcr", with_noise(mixed(640 << 10, 525), [(300_000, 6000)], 526), (8192, 4096, 768, 256),
                (1, 2, 3, 4), O.FIXED_MARKER, True))
    out.append(("mixed_g768", mixed(900 << 10, 527), (6144, 3072, 768), (1, 2, 3, 4), O.FIXED_MARKER, False))
    # random bytes behind a cascade: the true chain, re-entered in that segment, stops in them at a position its
    # speculative chain does not visit, and the speculative chain stops at one the true chain skips
    base = cascade(320 << 10, 531)
    out.append(("cascade_noise_strict", with_noise(base, [(140_000, 2500)], 533), REF, (1, 2, 3, 4), O.FIXED_MARKER,
                False))
    out.append(("cascade_noise_small", with_noise(base, [(164_400, 2500)], 533), SMALL, (1, 2, 3, 4), O.FIXED_MARKER,
                False))
    return out


def edge_cases():
    """(name, data, cands, methods, marker, pcr): file ends, candidate lists, markers and method subsets"""
    out = []
    seg_ref, seg_small = SEGU * 1024, SEGU * 512
    out.append(("n_lt_g_ref", inputs.text(700, 541), REF, (1, 2, 3, 4), O.FIXED_MARKER, False))
    out.append(("n_lt_g_small", inputs.log(300, 542), SMALL, (1, 2, 3, 4), O.FIXED_MARKER, True))
    for d in (-1, 0, 1):
        out.append(("n_2seg%+d_ref" % d, mixed(2 * seg_ref + d, 543 + d), REF, (1, 2, 3, 4), O.FIXED_MARKER, False))
        out.append(("n_3seg%+d_small" % d, mixed(3 * seg_small + d, 546 + d), SMALL, (1, 2, 3, 4), O.FIXED_MARKER, d == 1))
    # a last segment shorter than the smallest candidate
    out.append(("short_last_seg_ref", mixed(2 * seg_ref + 300, 550), REF, (1, 2, 3, 4), O.FIXED_MARKER, False))
    out.append(("short_last_seg_small", mixed(3 * seg_small + 200, 551), SMALL, (1, 2, 3, 4), O.FIXED_MARKER, True))
    # 16384 clamps to the last 7000 bytes and is the only candidate that can take them in one package
    out.append(("clamp_16384", inputs.text(2 * seg_ref + 7000, 552), (16384, 4096, 1024), (1, 2, 3, 4), O.FIXED_MARKER,
                False))
    # 16 distinct sizes once clamped to 8192 (the most the library takes)
    out.append(("sizes16", mixed(200 << 10, 553), (65536, 16384) + tuple(256 * k for k in range(32, 16, -1)),
                (1, 2, 3, 4), O.FIXED_MARKER, False))
    # markers of 1 to 4 bytes: package overheads of 15 to 18 bytes move the ratio compare
    for mb, marker in enumerate((b"\xfe", b"\x5a\xa5", b"\xfe\xfd\xfc", b"\x01\x02\x03\xfe"), 1):
        out.append(("marker%d" % mb, mixed(300 << 10, 560 + mb), SMALL, (1, 2, 3, 4), marker, mb % 2 == 0))
    out.append(("methods_1_3", mixed(400 << 10, 565, ("runs", "lowcard", "text")), REF, (1, 3), O.FIXED_MARKER, False))
    out.append(("methods_2_4", mixed(400 << 10, 566, ("text", "binrec", "csv")), SMALL, (2, 4), O.FIXED_MARKER, True))
    return out


def coverage(models):
    """the branches of the stitch and the file ends that the given [(name, Model)] reach on their true chains"""
    cov = set()
    for name, M in models:
        n = M.n
        true_pos = M.true_positions()
        if len(M.rounds) >= 60 and M.reentries and not any(f.merged for _, _, f in M.reentries):
            cov.add("cascade_g%d" % M.g)
        for sg, e in M.entries:
            sp = M.spec[sg]
            if e != sg * M.seglen:
                f = M.fix[sg]
                if f.merged and f.recs:
                    cov.add("merge_after_%s" % (len(f.recs) if len(f.recs) < 3 else "3+"))
                if M.pcr and any(r[2] == 255 for r in f.recs):
                    cov.add("pcr_raw_in_reentry")
                if not f.merged and f.stop is not None and f.stop not in {r[0] for r in sp.recs} and f.stop != sp.stop:
                    cov.add("strict_stop_in_reentry")
            if sp.stop is not None and sp.stop not in true_pos and sp.stop < M.raw_from:
                cov.add("spec_stop_skipped")
        for sg in range(1, M.n_seg):
            s0 = sg * M.seglen
            if s0 in true_pos:
                cov.add("exit_at_next_start")
            elif s0 < M.raw_from:
                cov.add("exit_past_next_start")
        r = n % M.seglen
        if n < M.g:
            cov.add("n_lt_g")
        if n >= M.seglen:
            cov.add({0: "n_k_seg", 1: "n_k_seg+1", M.seglen - 1: "n_k_seg-1"}.get(r, "n_other"))
        if 0 < r < M.cmin:
            cov.add("last_seg_short")
        cov.add("g%d" % M.g)
    return cov


WANT_COVERAGE = {"cascade_g1024", "cascade_g512", "merge_after_1", "merge_after_2", "merge_after_3+", "pcr_raw_in_reentry",
                 "strict_stop_in_reentry", "spec_stop_skipped", "exit_at_next_start", "exit_past_next_start", "n_lt_g",
                 "n_k_seg", "n_k_seg+1", "n_k_seg-1", "last_seg_short", "g1024", "g512", "g256", "g768"}


_MODELS = {}


def case_models():
    """[(name, data, cands, methods, marker, pcr, Model)] of large_cases() and edge_cases(), built once per process"""
    if not _MODELS:
        for name, data, cands, methods, marker, pcr in large_cases() + edge_cases():
            _MODELS[name] = (name, data, cands, methods, marker, pcr, model(data, cands, methods, marker, pcr))
    return list(_MODELS.values())


@pytest.mark.parametrize("pcr", [False, True])
def test_model_matches_oracle_on_dynamic_cases(pcr):
    for name, data, cfg in inputs.dynamic_cases():
        cands, methods = cfg["chunk_size"], tuple(cfg.get("method_ids", (1, 2, 3, 4)))
        M = model(data, cands, methods, pcr=pcr)
        assert M.packages == [tuple(p) for p in O.compress_body(data, cands, methods, per_chunk_raw=pcr)[1]], name


def test_model_matches_oracle_on_large_inputs():
    for name, data, cands, methods, marker, pcr, M in case_models():
        _, want = O.compress_body(data, cands, methods, marker, pcr)
        assert M.packages == [tuple(p) for p in want], name
        assert len(M.rounds) <= M.n_seg + 2, name


def test_cases_reach_every_branch_of_the_stitch():
    """the cases reach every branch and file end they were built for; a seed change that loses one fails here"""
    cases = case_models()
    models = [(c[0], c[-1]) for c in cases]
    cov = coverage(models)
    assert {len(c[4]) for c in cases} == {1, 2, 3, 4}
    assert {(1, 3), (2, 4)} <= {tuple(c[3]) for c in cases}
    assert WANT_COVERAGE <= cov, sorted(WANT_COVERAGE - cov)
    assert max(len(M.rounds) for _, M in models if M.g == 1024) >= 60
    assert max(M.n_seg for _, M in models if M.g == 512) > max(M.n_seg for _, M in models if M.g == 1024)


def test_model_cascade_resolves_one_segment_per_round():
    M = next(c[-1] for c in case_models() if c[0] == "cascade_ref_4M")
    assert M.n_seg == 64 and len(M.rounds) == 63
    assert all(len(r) == 1 for r in M.rounds) and not any(f.merged for _, _, f in M.reentries)
