"""A model of the multi-candidate ("dynamic") mode split across ranks, in plain Python over the CPU oracle.

Every rank holds one input range [lo, hi) of whole segments (distributed.dyn_shard_ranges) and runs
ambc_dyn_range_walk: the speculative walk of its segments, the stitch of the chain from lo, and in the first re-entry
launch the walks of every other position the chain can enter the range at (lo + k * g, k * g < min(8192, cands[0])),
each until it meets segment 0's speculative chain.  distributed.fold_dyn_entries follows the chain through the entry
tables; a rank whose true entry left segment 0 without meeting stitches it further (ambc_dyn_range_resolve) and the
tables are gathered again.  `RangeModel` restates compress.cu's bookkeeping on the walks of test_cpu_dynamic_walk's
`_walk`, so that the GPU tests can hold the library to the launches it took; the concatenated chains must be the
oracle's package list."""
import pytest

import inputs
import oracle as O
import test_cpu_dynamic_walk as W
from adaptive_compression_b200 import _lib as L
from adaptive_compression_b200 import distributed as D

WORLDS = (1, 2, 3, 5, 8, 17)
NATIVE = (1, 2, 3, 4)


class RangeModel:
    """one rank: spec[sg] (local segments), fix[sg] (latest re-entered Chain), rounds (item lists of every re-entry
    launch, candidates included), cands[k] (the walk from entry lo + k * g, k >= 1), table rows as the library's"""

    def __init__(self, data, cands, methods, marker, pcr, lo, hi, walk):
        self.n, self.lo, self.hi = len(data), lo, hi
        self.cands, self.pcr = cands, pcr
        self.g = W.gcd_of(cands)
        self.seglen = W.SEGU * self.g
        self.native = bool(set(methods) & set(NATIVE))
        rlen = hi - lo
        self.n_seg = -(-(-(-rlen // self.g)) // W.SEGU)
        self.bounds = [(lo + s * self.seglen, min(hi, lo + (s + 1) * self.seglen)) for s in range(self.n_seg)]
        self.walk = walk
        self.rounds, self.fix, self.cand = [], {}, {}
        self.resolved = set()
        n_e = min(min(8192, cands[0]) // self.g, -(-rlen // self.g)) if lo else min(1, rlen)
        self.entries = [lo + k * self.g for k in range(n_e)]
        self.table = []
        self._fill_table(data, cands, methods, marker, pcr, n_e)
        self.table0 = list(self.table)  # before any resolve

    def _fill_table(self, data, cands, methods, marker, pcr, n_e):
        lo, hi, walk = self.lo, self.hi, self.walk
        if not n_e:
            return
        if not self.native:
            for e in self.entries:
                if not pcr:
                    self.table.append((e, L.DYN_STOP, None, e))
                else:
                    cmin = cands[-1]
                    self.table.append((e, L.DYN_LEAVE, min(self.n, e + -(-(hi - e) // cmin) * cmin), None))
            return
        self.spec = [walk(s0, s1) for s0, s1 in self.bounds]
        extra = [(0, e) for e in self.entries[1:]]
        ex, st = self.stitch(lo, extra)
        for k, e in enumerate(self.entries):
            c = self.cand.get(k)
            if k == 0 or c.merged:
                self.table.append((e, L.DYN_JOIN, ex if st is None else None, st))
            elif c.stop is not None:
                self.table.append((e, L.DYN_STOP, None, c.stop))
            elif c.exit >= hi:
                self.table.append((e, L.DYN_LEAVE, c.exit, None))
            else:
                self.table.append((e, L.DYN_UNRESOLVED, c.exit, None))

    def follow(self, e):
        lst, stop = [], None
        for sg, (s0, s1) in enumerate(self.bounds):
            if e >= self.hi:
                break
            if e >= s1:
                continue
            sp = self.spec[sg]
            if e == s0:
                if sp.stop is not None:
                    stop = sp.stop
                    break
                e = sp.exit
                continue
            f = self.fix.get(sg)
            if f is not None and f.entry == e:
                last = sp if f.merged else f
                if last.stop is not None:
                    stop = last.stop
                    break
                e = last.exit
                continue
            lst.append((sg, e))
            if sp.stop is not None:
                stop = sp.stop
                break
            e = sp.exit
        return lst, e, stop

    def stitch(self, e0, extra=()):
        first = True
        while True:
            lst, ex, st = self.follow(e0)
            items = lst + (list(extra) if first else [])
            if not items:
                return ex, st
            assert len(self.rounds) <= 2 * self.n_seg + 4, "the stitch does not settle"
            self.rounds.append(items)
            for i, (sg, e) in enumerate(items):
                f = self.walk(e, self.bounds[sg][1], sg)
                if i < len(lst):
                    self.fix[sg] = f
                else:
                    self.cand[self.entries.index(e)] = f
            first = False

    def row(self, entry):
        return next(t for t in self.table if t[0] == entry)

    def resolve(self, entry):
        k = self.entries.index(entry)
        t = self.table[k]
        if t[1] == L.DYN_UNRESOLVED:
            ex, st = self.stitch(t[2])
            self.table[k] = (entry, L.DYN_STOP, None, st) if st is not None else (entry, L.DYN_LEAVE, ex, None)
            self.resolved.add(k)
        return self.table[k]

    def chain(self, entry):
        """-> (records [(pos, size, type, comp)], stop or None) of the chain from the true entry"""
        if entry >= self.hi:
            return [], None
        if not self.native:
            if not self.pcr:
                return [], entry
            cmin, recs, p = self.cands[-1], [], entry
            while p < self.hi:
                s = min(cmin, self.n - p)
                recs.append((p, s, 255, s))
                p += s
            return recs, None
        k = self.entries.index(entry)
        recs, e, on_spec = [], entry, False
        if k:
            c = self.cand[k]
            recs += c.recs
            if c.merged:
                e, on_spec = c.exit, True
            elif c.stop is not None:
                return recs, c.stop
            elif c.exit >= self.hi:
                return recs, None
            else:
                assert k in self.resolved
                e = c.exit
        for sg, (s0, s1) in enumerate(self.bounds):
            if e >= self.hi:
                break
            if e >= s1:
                continue
            sp, frm = self.spec[sg], 0
            if e != s0 and on_spec:
                frm = [r[0] for r in sp.recs].index(e)
            elif e != s0:
                f = self.fix[sg]
                assert f.entry == e
                recs += f.recs
                if f.merged:
                    frm = [r[0] for r in sp.recs].index(f.exit)
                else:
                    if f.stop is not None:
                        return recs, f.stop
                    e = f.exit
                    continue
            on_spec = False
            recs += sp.recs[frm:]
            if sp.stop is not None:
                return recs, sp.stop
            e = sp.exit
        return recs, None

    def walk_launches(self):
        return (1 + len(self.rounds)) if (self.native and self.entries) else 0


class Sharded:
    """R ranks: models, fold rounds, the true entries, the stop, the concatenated chain"""

    def __init__(self, data, cands, methods, marker, pcr, world, cache=None):
        data = bytes(data)
        cands = tuple(sorted({int(c) for c in cands}, reverse=True))
        self.n, self.world = len(data), world
        cache = {} if cache is None else cache
        g = W.gcd_of(cands)
        spec_pos = {}
        self.ranges = D.dyn_shard_ranges(self.n, cands, world)
        self.ranks = []
        for lo, hi in self.ranges:
            def walk(start, end, sg=None, _lo=lo):
                # sg given: a list-mode walk in local segment sg, stopped where it meets that segment's spec chain
                gs = None if sg is None else (_lo // (W.SEGU * g)) + sg
                key = (start, end, gs)
                if key not in cache:
                    vis = () if gs is None else spec_pos[gs]
                    cache[key] = W._walk(data, cands, methods, marker, pcr, start, end, vis)
                    if gs is None and start % (W.SEGU * g) == 0:
                        spec_pos[start // (W.SEGU * g)] = {r[0] for r in cache[key].recs}
                elif gs is None and start % (W.SEGU * g) == 0:
                    spec_pos[start // (W.SEGU * g)] = {r[0] for r in cache[key].recs}
                return cache[key]
            self.ranks.append(RangeModel(data, cands, methods, marker, pcr, lo, hi, walk))
        self.fold_rounds = 0
        self.stuck = []
        while True:
            self.fold_rounds += 1
            entries, stuck, stop = D.fold_dyn_entries([m.table for m in self.ranks], self.n)
            if stuck is None:
                break
            self.stuck.append(stuck)
            self.ranks[stuck].resolve(entries[stuck])
            assert self.fold_rounds <= world, "the fold does not settle within R rounds"
        self.entries, self.stop = entries, stop
        self.chains = [m.chain(e) if e is not None else ([], None) for m, e in zip(self.ranks, entries)]
        self.chain = [r for c, _ in self.chains for r in c]
        stops = [s for _, s in self.chains if s is not None]
        assert stops[:1] == ([stop] if stop is not None else [])

    @property
    def packages(self):
        out = [(t, size, comp) for _, size, t, comp in self.chain]
        if self.stop is not None and self.stop < self.n:
            out.append((255, self.n - self.stop, self.n - self.stop))
        return out


# ---- inputs for the rank boundaries ------------------------------------------------------------------------------
SEG_REF, SEG_SMALL = W.SEGU * 1024, W.SEGU * 512


def shard_cases():
    """(name, data, cands, methods, marker, pcr, worlds): inputs built for the rank boundaries"""
    out = []
    # random bytes right at the start of a range: strict stop at a rank's entry; later ranks inside the raw tail
    base = W.mixed(6 * SEG_SMALL, 601)
    out.append(("stop_at_boundary", W.with_noise(base, [(2 * SEG_SMALL, 9000)], 602), W.SMALL, NATIVE, O.FIXED_MARKER,
                False, WORLDS))
    # random bytes at the end of a range: the stop lies in the range's last segment
    out.append(("stop_in_last_seg", W.with_noise(base, [(3 * SEG_SMALL - 6000, 12000)], 603), W.SMALL, NATIVE,
                O.FIXED_MARKER, False, WORLDS))
    # per-chunk-raw pieces across boundaries (raw stretches around the cuts)
    out.append(("pcr_boundary", W.with_noise(base, [(2 * SEG_SMALL - 700, 3000), (4 * SEG_SMALL - 300, 2000)], 604),
                (8192, 2048, 1536), NATIVE, O.FIXED_MARKER, True, WORLDS))
    # no native method: one raw package, or per-chunk-raw pieces of cands[-1] that do not line up with the ranges
    out.append(("no_native_strict", W.mixed(3 * SEG_SMALL + 700, 605), W.SMALL, (), O.FIXED_MARKER, False, WORLDS))
    out.append(("no_native_pcr", W.mixed(3 * SEG_REF + 100, 606), (6144, 3072), (), O.FIXED_MARKER, True, WORLDS))
    # a last rank shorter than g, and shorter than S
    out.append(("last_lt_g", W.mixed(4 * SEG_SMALL + 300, 607), W.SMALL, NATIVE, O.FIXED_MARKER, False, (2, 4, 5)))
    out.append(("last_lt_S", W.mixed(4 * SEG_SMALL + 5000, 608), W.SMALL, NATIVE, O.FIXED_MARKER, False, (2, 4, 5)))
    # the cascade across every boundary: the fold needs R rounds
    out.append(("cascade_every", W.cascade(16 * SEG_SMALL, 609, 512), W.SMALL, NATIVE, O.FIXED_MARKER, False,
                (2, 3, 5, 8)))
    return out


_SHARDED = {}


def sharded_models():
    """[(name, world, data, cands, methods, marker, pcr, Sharded)]: the large and edge cases of test_cpu_dynamic_walk
    and shard_cases(), for every world size"""
    if not _SHARDED:
        cases = [c + (WORLDS,) for c in W.large_cases() + W.edge_cases()] + shard_cases()
        for name, data, cands, methods, marker, pcr, worlds in cases:
            cache = {}
            for R in worlds:
                S = Sharded(data, cands, methods, marker, pcr, R, cache)
                _SHARDED[(name, R)] = (name, R, data, cands, methods, marker, pcr, S)
    return list(_SHARDED.values())


def coverage(items):
    cov = set()
    for name, R, data, cands, methods, marker, pcr, S in items:
        n = S.n
        nonempty = [(lo, hi) for lo, hi in S.ranges if hi > lo]
        if len(nonempty) < R:
            cov.add("empty_ranks")
        if len(nonempty) > 1:
            llo, lhi = nonempty[-1]
            S_max = min(8192, max(cands))
            if lhi - llo < W.gcd_of(cands):
                cov.add("last_lt_g")
            elif lhi - llo < S_max:
                cov.add("last_lt_S")
        if S.fold_rounds == R and R >= 3 and len(S.stuck) == R - 1:
            cov.add("unresolved_every_boundary")
        if S.stuck:
            cov.add("unresolved")
        for r, (m, e) in enumerate(zip(S.ranks, S.entries)):
            if e is None:
                if m.hi > m.lo and S.stop is not None and m.lo > S.stop:
                    cov.add("rank_in_raw_tail")
                continue
            if r and e == m.lo:
                cov.add("exit_at_hi")
            k = m.entries.index(e) if e in m.entries else None
            if k and m.native:
                c = m.cand[k]
                if c.merged:
                    cov.add("merge_after_%s" % (len(c.recs) if len(c.recs) < 3 else "3+"))
                if c.stop is not None and not c.merged:
                    lo_chain = {x[0] for x in m.chain(m.lo)[0]}
                    if c.stop == e:
                        cov.add("stop_at_entry")
                    elif c.stop not in lo_chain:
                        cov.add("stop_in_candidate_skipped")
            recs, st = S.chains[r]
            if st is not None and m.n_seg > 1 and st >= m.bounds[-1][0]:
                cov.add("stop_in_last_segment")
            if pcr and any(p < m.hi < p + s and t == 255 for p, s, t, _ in recs):
                cov.add("pcr_across_boundary")
        cov.add("marker%d" % len(marker))
        cov.add("methods_" + "".join(str(x) for x in methods))
    return cov


WANT = {"empty_ranks", "last_lt_g", "last_lt_S", "unresolved", "unresolved_every_boundary", "rank_in_raw_tail",
        "exit_at_hi", "merge_after_1", "merge_after_2", "merge_after_3+", "stop_at_entry", "stop_in_candidate_skipped",
        "stop_in_last_segment", "pcr_across_boundary", "marker1", "marker2", "marker3", "marker4", "methods_13",
        "methods_24", "methods_"}


def test_sharded_chain_matches_oracle():
    bad = []
    for name, R, data, cands, methods, marker, pcr, S in sharded_models():
        _, want = O.compress_body(data, cands, methods, marker, pcr)
        if S.packages != [tuple(p) for p in want]:
            bad.append((name, R))
        if S.fold_rounds > R:
            bad.append((name, R, "rounds", S.fold_rounds))
    assert not bad, bad


def test_shard_cases_reach_every_boundary_branch():
    cov = coverage(sharded_models())
    assert WANT <= cov, sorted(WANT - cov)


def test_cascade_across_every_boundary_takes_R_rounds():
    for name, R, *_, S in sharded_models():
        if name == "cascade_every":
            ranks = sum(hi > lo for lo, hi in S.ranges)
            assert S.fold_rounds == ranks and S.stuck == list(range(1, ranks)), (R, S.stuck)


def test_one_rank_is_the_single_gpu_model():
    """R = 1: the range [0, n) walks, rounds and chain of test_cpu_dynamic_walk's model"""
    models = {c[0]: c[-1] for c in W.case_models()}
    for name, R, data, cands, methods, marker, pcr, S in sharded_models():
        if R != 1 or name not in models:
            continue
        M = models[name]
        assert S.ranks[0].walk_launches() == M.walk_launches(), name
        assert S.chain == M.chain, name


def test_dyn_fragment_plan_places_the_raw_tail_and_end():
    ranges = [(0, 100), (100, 200), (200, 250), (250, 250)]
    plan, body_len = D.dyn_fragment_plan([(40, -1), (30, 150), (0, -1), (0, -1)], ranges, 250, 4)
    ovh = 18
    assert plan == [(0, 40, "packed"), (40, 30 + ovh + 50, "raw_starts_here"), (40 + 30 + ovh + 50, 50, "in_raw_tail"),
                    (40 + 30 + ovh + 100, 16, "in_raw_tail")]
    assert body_len == 40 + 30 + ovh + 100 + 16
    plan, body_len = D.dyn_fragment_plan([(40, -1), (35, -1)], [(0, 100), (100, 180)], 180, 1)
    assert plan == [(0, 40, "packed"), (40, 35 + 13, "packed")] and body_len == 88
    with pytest.raises(L.AmbcError, match="4 GiB"):
        D.dyn_fragment_plan([(10, 5), (0, -1)], [(0, 1 << 31), (1 << 31, (1 << 32) + 10)], (1 << 32) + 10)


def test_dyn_shard_ranges_are_whole_segments():
    for n in (0, 1, 65535, 65536, 65537, 10 ** 6):
        for R in WORLDS:
            rs = D.dyn_shard_ranges(n, inputs.REF_DEFAULT_CANDIDATES, R)
            assert rs[0][0] == 0 and rs[-1][1] == n and len(rs) == R
            assert all(a[1] == b[0] for a, b in zip(rs, rs[1:]))
            assert all(lo % 65536 in (0, n % 65536) and hi % 65536 in (0, n % 65536) for lo, hi in rs)
            assert D.dyn_buffer_span(*rs[-1], n)[1] <= n
