"""Seeded chunks that sit on the decision boundaries of the chunk trial (sf_select in csrc/select_fast.cuh).

sf_select does not run the reference's selection rules (adaptive_compressor.py:537-590, the should_use gates of
compression_methods.py) literally: it restates them as integer predicates, decides the entropy gate in fp32 unless it
is close, and skips trials whose outcome is proven.  Corpus chunks almost never land on those boundaries, so this
module builds chunks that do, on both sides, for both instantiations (chunks of up to 4096 bytes run
k_select_fast<4096>, 4097..8192 run k_select_fast<8192>).

A case is (label, side, data, chunk, methods, marker): `data` is one chunk of `chunk` bytes (or a short last chunk
of a `chunk` grid), `side` says where it sits relative to the boundary the label names.  numbers() computes the
oracle's view of a chunk: the gate inputs, every method's payload length and the chosen (type, len).  Everything is
a function of fixed seeds; cases() builds the list once per process."""
from collections import namedtuple

import numpy as np

import inputs
import oracle as O

Case = namedtuple("Case", "label side data chunk methods marker")

MARKERS = {1: b"\xfe", 2: b"\x5a\xa5", 3: b"\xfe\xfd\xfc", 4: O.FIXED_MARKER}
NATIVE = (1, 2, 3, 4)
RANGE = {1: (32, 4096), 2: (128, 8192), 3: (32, 8192), 4: (32, 4096)}  # adaptive_compressor.py:114-127


def inst(n):
    """the k_select_fast instantiation that runs a chunk of n bytes"""
    return 4096 if n <= 4096 else 8192


# ---- the oracle's numbers ------------------------------------------------------------------------------------------
def rle_rep(a):
    """(rep, ss) of the RLE gate: sampled positions i with a[i] == a[i + 1] (compression_methods.py:154-180)"""
    n = len(a)
    ss = min(1000, n)
    step = max(1, n // ss) if n >= 4 else 1
    i = np.arange(0, n - 1, step)
    return int((a[i] == a[i + 1]).sum()), ss


def distinct3(a):
    """distinct 3-byte slices among the first min(n - 3, min(1000, n)) positions (compression_methods.py:315-343)"""
    n = len(a)
    cnt = min(n - 3, min(1000, n))
    if cnt <= 0:
        return 0
    t = a[:cnt].astype(np.int64) | (a[1:cnt + 1].astype(np.int64) << 8) | (a[2:cnt + 2].astype(np.int64) << 16)
    return int(np.unique(t).size)


def lz_min(n):
    """sf_lz_lower_bound: the smallest Dictionary payload of n bytes"""
    r = (n - 1) % 32
    return 2 + 4 * ((n - 1) // 32) + min(2 * r, 4)


def hf_min(n):
    """the smallest Huffman payload of n bytes (two symbols, one bit each)"""
    return 1 + 5 * 2 + 4 + (n + 7) // 8


def lz_tokens(payload):
    """Dictionary payload -> [(position, length, token bytes)] (literal: 0, byte; match: 1, d lo, d hi, length)"""
    out, p, i = [], 0, 0
    while i < len(payload):
        if payload[i] == 0:
            out.append((p, 1, 2)); p += 1; i += 2
        else:
            L = payload[i + 3]
            out.append((p, L, 4)); p += L; i += 4
    return out


def staged_checks(payload, n):
    """[(rest, lb)] after the first two stages of sf_lz_parse's staged parse (n >= 1024), from the oracle's tokens"""
    toks = lz_tokens(payload)
    out, total, k = [], 0, 0
    for b in ((11 * n // 32) & ~31, (9 * n // 16) & ~31):
        while k < len(toks) and toks[k][0] < b:
            total += toks[k][2]; k += 1
        entry = toks[k][0] if k < len(toks) else n
        rest = n - entry
        out.append((rest, total + (4 * (rest >> 5) + min(4, 2 * (rest & 31)) if rest > 0 else 0)))
    return out


def ngram_bound(a, hashed=False):
    """(4 D + 2 F) / 3 of sf_lz_bound_ngrams: D = distinct 4-grams at the positions p < n - 3, F = positions
    2 <= p < n - 3 whose trigram and the trigrams at p - 1 and p - 2 occur there first.  hashed=True restates the
    kernel's own count: D as the occupied bits of a 2^17-bit set of hashed 4-grams, "first" as the minimum position
    per 12-bit trigram hash (both can only lose some of D and F)"""
    n = len(a)
    if n < 4:
        return 0
    a64 = a.astype(np.uint64)
    g4 = a64[:n - 3] | (a64[1:n - 2] << 8) | (a64[2:n - 1] << 16) | (a64[3:] << 24)
    g3 = a64[:n - 2] | (a64[1:n - 1] << 8) | (a64[2:] << 16)
    if hashed:
        D = int(np.unique(((g4 * 2654435761) & 0xFFFFFFFF) >> 15).size)
        key = ((g3 * 2654435761) & 0xFFFFFFFF) >> 20
    else:
        D = int(np.unique(g4).size)
        key = g3
    _, first_pos = np.unique(key, return_index=True)
    f = np.zeros(n - 2, dtype=bool)
    f[first_pos] = True
    F = int((f[2:n - 3] & f[1:n - 4] & f[:n - 5]).sum()) if n > 5 else 0
    return (4 * D + 2 * F) // 3


def numbers(data, methods=NATIVE, marker=O.FIXED_MARKER):
    """the oracle's numbers of one chunk: gate inputs, should_use, payload lengths, chosen (type, len)"""
    a = np.frombuffer(bytes(data), dtype=np.uint8)
    n = len(a)
    rep, ss = rle_rep(a)
    d3 = distinct3(a)
    K = int(np.unique(a).size)
    H = O.entropy(data) if n else 0.0
    pay, gate = {}, {}
    for m in (1, 2, 3):
        gate[m] = O.should_use(m, data)
        p = O.compress(m, data, lz_fast=True)
        pay[m] = len(p) if isinstance(p, bytes) else None
    ovh = len(marker) + 14
    best, bt = 1.0, 255
    for m in methods:  # adaptive_compressor.py:565-579 for one candidate
        lo, hi = RANGE[m]
        if not (lo <= n <= hi) or not O.should_use(m, data):
            continue
        cl = n if m == 4 else pay[m]
        if cl is None:
            continue
        r = (cl + ovh) / n
        if r < best:
            best, bt = r, m
    chosen = (bt, n if bt == 255 else (n if bt == 4 else pay[bt]))
    return dict(n=n, rep=rep, ss=ss, distinct3=d3, K=K, H=H, pay=pay, gate=gate, ovh=ovh, chosen=chosen)


# ---- construction helpers ------------------------------------------------------------------------------------------
def from_eq(eq, rng, values=256):
    """bytes whose neighbour equalities are exactly eq (length n - 1); every new run gets a random other value"""
    n = len(eq) + 1
    out = np.empty(n, dtype=np.uint8)
    out[0] = rng.randint(values)
    for i in range(n - 1):
        if eq[i]:
            out[i + 1] = out[i]
        else:
            v = rng.randint(values - 1)
            out[i + 1] = v + (v >= out[i])
    return out


def runs_data(n, R, rng, min_len=1, max_len=255, values=256, all_values=True):
    """n bytes in exactly R runs of random values (neighbours differ), lengths in [min_len, max_len]"""
    assert R * min_len <= n <= R * max_len
    lens = np.full(R, min_len, dtype=np.int64)
    left = n - R * min_len
    while left:
        i = rng.randint(R)
        if lens[i] < max_len:
            lens[i] += 1; left -= 1
    vals = np.empty(R, dtype=np.int64)
    if all_values and R >= values:
        order = rng.permutation(R)[:values]  # every value at least once (K = 256 shuts the Huffman gate)
        vals[:] = -1
        vals[order] = np.arange(values)
    else:
        vals[:] = -1
    for i in range(R):
        if vals[i] < 0 or (i and vals[i] == vals[i - 1]):
            while True:
                v = rng.randint(values)
                if (i == 0 or v != vals[i - 1]) and (i + 1 >= R or v != vals[i + 1]):
                    break
            vals[i] = v
    for i in range(1, R):  # (a value placed above may still equal its predecessor)
        while vals[i] == vals[i - 1]:
            vals[i] = (vals[i] + 1 + rng.randint(values - 1)) % values
    return np.repeat(vals.astype(np.uint8), lens)


def search(a, f, target, rng, lo=0, hi=None, steps=4000, move=None, ok=None):
    """seeded local search: mutate one byte of a[lo:hi] at a time and keep the mutation if |f - target| does not
    grow (and ok() holds).  -> (array, f) of the closest state reached"""
    a = a.copy()
    hi = len(a) if hi is None else hi
    cur = f(a)
    for _ in range(steps):
        if cur == target:
            break
        p = lo + rng.randint(hi - lo)
        old = a[p]
        if move is None:
            a[p] = a[rng.randint(len(a))]
        else:
            move(a, p, rng)
        if a[p] == old:
            continue
        v = f(a)
        if v is not None and abs(v - target) <= abs(cur - target) and (ok is None or ok(a)):
            cur = v
        else:
            a[p] = old
    return a, cur


def plen(m, a):
    p = O.compress(m, a.tobytes(), lz_fast=True)
    return len(p) if isinstance(p, bytes) else None


def _by_counts(counts, rng):
    """a random permutation of the multiset {symbol: count}"""
    a = np.repeat(np.array(list(counts.keys()), dtype=np.uint8), list(counts.values()))
    return a[rng.permutation(a.size)]


# ---- families --------------------------------------------------------------------------------------------------------
def rle_gate():
    """10 rep - 3 (ss - 1) on both sides of 0 (= 0 where n - 1 is a multiple of 10 and n < 1000): the sampled
    positions (steps 1..8, the step-4 mask) carry exactly rep equal neighbours, every other position repeats its
    predecessor (so that the open gate leads to an RLE winner where the step allows it)"""
    out = []
    rng = np.random.RandomState(1101)
    for n in (32, 33, 100, 101, 991, 999, 1000, 1001, 1999, 2000, 2001, 3000, 3999, 4000, 4096,
              4097, 5000, 6000, 7000, 8192):
        ss = min(1000, n)
        step = max(1, n // ss)
        thr = 3 * (ss - 1)
        samp = np.arange(0, n - 1, step)
        r_open = thr // 10 + 1
        reps = [r_open - 1, r_open] + ([r_open - 2] if thr % 10 == 0 else [])
        for rep in reps:
            eq = np.ones(n - 1, dtype=bool)
            eq[samp] = False
            eq[rng.choice(samp, rep, replace=False)] = True
            out.append(Case("rle_gate", 10 * rep - thr, from_eq(eq, rng).tobytes(), n, NATIVE, O.FIXED_MARKER))
    return out


def dict_gate():
    """10 distinct3 - 8 min(1000, n) on both sides of 0 (= 0 where 8 min(1000, n) is a multiple of 10): a random
    period of a bytes has exactly a distinct trigrams"""
    out = []
    rng = np.random.RandomState(1201)
    for n in (128, 129, 999, 1000, 1002, 1003, 4096, 8192):
        ss = min(1000, n)
        thr = 8 * ss
        a_open = (thr - 1) // 10
        for per in sorted({a_open, a_open + 1, thr // 10 + 1 if thr % 10 == 0 else a_open}):
            out.append(Case("dict_gate", 10 * per - thr, periodic(n, per, rng).tobytes(), n, NATIVE, O.FIXED_MARKER))
    return out


def periodic(n, per, rng, values=256):
    """n bytes of period per whose per trigrams (wrap included) are all distinct"""
    while True:
        r = rng.randint(values, size=per).astype(np.uint8)
        a = np.resize(r, n)
        w = np.resize(r, per + 2)
        t = w[:per].astype(np.int64) | (w[1:per + 1].astype(np.int64) << 8) | (w[2:].astype(np.int64) << 16)
        if np.unique(t).size == per:
            return a


def huff_gate():
    """K in {1, 2, 255, 256}, n in {99, 100}, entropy exactly 7 (dyadic), inside the fp64 window on both sides of 7,
    and just outside +-0.02; Huffman is the only method, so the gate alone decides"""
    out = []
    rng = np.random.RandomState(1301)
    M3 = (3,)
    for n in (100, 4096, 8192):
        for K in (1, 2, 255, 256):
            if K > n:
                continue
            cnt = {s: 1 for s in range(K)}
            cnt[0] = n - (K - 1)  # skewed: entropy well below 7
            if K == 2:
                cnt = {7: n // 2 + 3, 200: n - n // 2 - 3}
            out.append(Case("huff_K", K, _by_counts(cnt, rng).tobytes(), n, M3, O.FIXED_MARKER))
    for n in (99, 100):
        a = rng.choice(np.array([3, 9], dtype=np.uint8), size=n)
        out.append(Case("huff_n", n, a.tobytes(), n, M3, O.FIXED_MARKER))
        out.append(Case("huff_n", n, a.tobytes(), n, NATIVE, O.FIXED_MARKER))
    # exactly 7.0: 128 x (n / 128), and 32 x (n / 64) + 128 x (n / 256)
    for n in (4096, 8192):
        out.append(Case("huff_H7", 0, _by_counts({s: n // 128 for s in range(128)}, rng).tobytes(), n, M3, O.FIXED_MARKER))
        c = {s: n // 64 for s in range(32)}
        c.update({32 + s: n // 256 for s in range(128)})
        out.append(Case("huff_H7", 0, _by_counts(c, rng).tobytes(), n, M3, O.FIXED_MARKER))
    # near 7, both sides, inside the fp64 window and just outside +-0.02
    for n in (4096, 8192):
        for tgt, side in ((7.0, -1), (7.0, 1), (6.98, -2), (7.02, 2)):
            a = near_entropy(n, tgt, side, rng)
            out.append(Case("huff_near7", side, a.tobytes(), n, M3, O.FIXED_MARKER))
    return out


def _H(counts, n):
    p = counts[counts > 0] / n
    return float(-(p * np.log2(p)).sum())


def near_entropy(n, tgt, side, rng, steps=3000):
    """move single counts between the symbols of a dyadic histogram (32 x n/64 + 128 x n/256, entropy 7) until the
    entropy is as close to tgt as the search gets, strictly on the given side of 7 (|side| = 2: beyond tgt, outside
    the fp32 path's window)"""
    c = np.zeros(256, dtype=np.int64)
    c[:32] = n // 64
    c[32:160] = n // 256
    want = (lambda h: h < 7.0 and (side == -1 or h < tgt)) if side < 0 else (lambda h: h > 7.0 and (side == 1 or h > tgt))
    score = lambda h: (not want(h), abs(h - tgt))  # noqa: E731
    cur = score(_H(c, n))
    for _ in range(steps):
        i, j = rng.randint(160), rng.randint(160)
        if i == j or c[i] <= 1:
            continue
        c[i] -= 1; c[j] += 1
        s = score(_H(c, n))
        if s <= cur:
            cur = s
        else:
            c[i] += 1; c[j] -= 1
    while True:  # the exact (first-occurrence order) entropy of the permuted chunk decides the side
        a = _by_counts({s: int(c[s]) for s in range(256) if c[s]}, rng)
        h = O.entropy(a.tobytes())
        if want(h):
            return a


def dict_huff_ties():
    """Dictionary - Huffman in {-1, 0, +1} (the Dictionary payload wins ties with Huffman: cutoff = hf_len + 1),
    searched from text and log chunks by one-byte mutations"""
    out = []
    rng = np.random.RandomState(1401)
    f = lambda a: None if (plen(2, a) is None or plen(3, a) is None) else plen(2, a) - plen(3, a)  # noqa: E731
    for kind in ("text", "log"):
        for n in (4096, 8192):
            a = np.frombuffer(inputs.make(kind, n, 1402 + n), dtype=np.uint8)
            for tgt in (0, -1, 1):
                a, v = search(a, f, tgt, rng, lo=1003)
                if v == tgt:
                    out.append(Case("dict_huff", v, a.tobytes(), n, NATIVE, O.FIXED_MARKER))
    return out


def rle_huff_ties():
    """RLE - Huffman in {-1, 0, +1} on three-symbol runs (counts fix the Huffman payload: 20 + ceil((n + c2 + c3) / 8),
    the number of runs R fixes RLE's 2 R), RLE and Huffman only"""
    out = []
    rng = np.random.RandomState(1501)
    n = 4096
    for m in (1000, 1008):  # c2 + c3: Huffman payloads 657 (odd) and 658 (even)
        hf = 20 + -(-(n + m) // 8)
        for R in sorted({(hf - 1) // 2, (hf + 1) // 2, hf // 2}):
            a = three_runs(n, R, (n - m, 600, m - 600), rng)
            out.append(Case("rle_huff", 2 * R - hf, a.tobytes(), n, (1, 3), O.FIXED_MARKER))
            out.append(Case("rle_huff", 2 * R - hf, a.tobytes(), n, (1, 2, 3), O.FIXED_MARKER))
    return out


def three_runs(n, R, counts, rng):
    """R runs over symbols (a, b, a, c, ...) with the given symbol counts"""
    sym = [0 if i % 2 == 0 else (1 if i % 4 == 1 else 2) for i in range(R)]
    vals = np.array([17, 90, 201], dtype=np.uint8)
    lens = np.zeros(R, dtype=np.int64)
    for s in range(3):
        idx = [i for i in range(R) if sym[i] == s]
        k = len(idx)
        cut = np.sort(rng.choice(np.arange(1, counts[s]), k - 1, replace=False)) if k > 1 else np.array([], dtype=np.int64)
        lens[idx] = np.diff(np.concatenate([[0], cut, [counts[s]]]))
    assert lens.min() >= 1 and lens.max() <= 255 and lens.sum() == n
    return np.repeat(vals[sym], lens)


def rle_dict_ties():
    """RLE - Dictionary in {-2, 0, +2} (both payloads are even; RLE wins ties), RLE and Dictionary only: runs of a
    random period, tuned by one-byte mutations"""
    out = []
    rng = np.random.RandomState(1601)
    f = lambda a: None if (plen(1, a) is None or plen(2, a) is None) else plen(1, a) - plen(2, a)  # noqa: E731
    n = 4096
    per = runs_data(256, 16, rng, all_values=False)
    base = np.resize(per, n)
    for tgt in (0, -2, 2):
        base, v = search(base, f, tgt, rng, lo=300, ok=lambda a: O.should_use(1, a.tobytes()) and O.should_use(2, a.tobytes()))
        if v == tgt:
            out.append(Case("rle_dict", v, base.tobytes(), n, (1, 2), O.FIXED_MARKER))
            out.append(Case("rle_dict", v, base.tobytes(), n, NATIVE, O.FIXED_MARKER))
    return out


def rle_shortcut():
    """RLE payload == sf_lz_lower_bound(n) (methods 1, 2) and == the smallest Huffman payload (methods 1, 3), +-2: the
    outright RLE win at equality"""
    out = []
    rng = np.random.RandomState(1701)
    for n in (4096, 2000):
        for d in (-2, 0, 2):
            R = (lz_min(n) + d) // 2
            out.append(Case("rle_eq_lzmin", d, runs_data(n, R, rng, all_values=False).tobytes(), n, (1, 2), O.FIXED_MARKER))
    for n in (4088, 2008):  # hf_min even
        for d in (-2, 0, 2):
            R = (hf_min(n) + d) // 2
            a = runs_data(n, R, rng, all_values=False, values=2)
            out.append(Case("rle_eq_hfmin", d, a.tobytes(), n, (1, 3), O.FIXED_MARKER))
    return out


def benefit():
    """best + ovh - n in {-1, 0, +1} for package overheads 15..18 (markers of 1..4 bytes), with RLE-only chunks
    (runs of random values, all 256 values, >= 80 % distinct trigrams), and Huffman-only and Dictionary-only chunks
    reached by search"""
    out = []
    rng = np.random.RandomState(1801)
    for n in (4096, 4095):
        for P in range(n - 19, n - 13):
            if P % 2:
                continue
            a = runs_data(n, P // 2, rng, min_len=1, max_len=4)
            for mb, mk in MARKERS.items():
                g = P + mb + 14 - n
                if abs(g) <= 1:
                    out.append(Case("benefit_rle", g, a.tobytes(), n, NATIVE, mk))
    # Huffman only: ~200 symbols at entropy ~6 (the Dictionary gate shut by distinct trigrams, RLE by no repeats)
    for n in (4096, 8192):
        K = 200 if n == 4096 else 240
        f = lambda x: plen(3, x)  # noqa: E731
        best = None
        for s_ in np.linspace(0.5, 40.0, 80):  # the skew whose Huffman payload lies closest to n - 16
            w = np.exp(-np.arange(K) / (K / s_))
            x = rng.choice(K, size=n, p=w / w.sum()).astype(np.uint8)
            v = f(x)
            if v is not None and (best is None or abs(v - (n - 16)) < abs(best[0] - (n - 16))):
                best = (v, x)
        a = best[1]
        for P in range(n - 19, n - 13):
            a, v = search(a, f, P, rng, move=lambda x, p, r: x.__setitem__(p, r.randint(K)))
            if v == P and not O.should_use(1, a.tobytes()) and not O.should_use(2, a.tobytes()):
                for mb, mk in MARKERS.items():
                    g = P + mb + 14 - n
                    if abs(g) <= 1:
                        out.append(Case("benefit_huff", g, a.tobytes(), n, NATIVE, mk))
    # Dictionary only: a random period of 600 bytes over all 256 values (Huffman shut by K = 256), then random bytes
    for n in (4096, 4095, 8192, 8191):
        a = np.resize(np.concatenate([rng.permutation(256), rng.randint(256, size=344)]).astype(np.uint8), n)
        tail = n // 3
        a[-tail:] = rng.randint(256, size=tail)
        f = lambda x: plen(2, x)  # noqa: E731
        for P in range(n - 19, n - 13):
            if P % 2:
                continue
            a, v = search(a, f, P, rng, lo=1003, move=lambda x, p, r: x.__setitem__(p, x[p - 600] if r.rand() < 0.5 else r.randint(256)),
                          ok=lambda x: not O.should_use(1, x.tobytes()))
            if v == P:
                for mb, mk in MARKERS.items():
                    g = P + mb + 14 - n
                    if abs(g) <= 1:
                        out.append(Case("benefit_dict", g, a.tobytes(), n, NATIVE, mk))
    return out


def staged():
    """the staged parse (n >= 1024, a Huffman payload in hand, 100 distinct3 >= 34 min(1000, n)): its threshold
    (distinct3 = 339 / 340) and its abort bound at the second stage boundary, where rest % 32 == 0 and every token
    behind it is an exact 32-byte match (the bound is tight): Dictionary payload = Huffman payload (the Dictionary
    wins: cutoff - 1) and Huffman payload + 1 (it loses: = cutoff)"""
    out = []
    rng = np.random.RandomState(1901)
    for n in (4096,):  # (the search does not reach the 8192-byte version within its budget)
        b2 = (9 * n // 16) & ~31
        for per in (339, 340):
            for tgt in (0, 1):
                a = staged_chunk(n, per, b2, tgt, rng)
                if a is not None:
                    out.append(Case("staged", (per, tgt), a.tobytes(), n, NATIVE, O.FIXED_MARKER))
    return out


def staged_chunk(n, per, b, tgt, rng, tries=3, D=2048):
    """first 1003 bytes: period per over 40 symbols (distinct3 = per, entropy < 7); [1003, b - 8): literals and
    copies, tuned; [b - 8, b): random; [b, n): a copy from distance D (32-byte matches to the end)"""
    for _ in range(tries):
        a = np.empty(n, dtype=np.uint8)
        a[:1003] = periodic(1003, per, rng, values=40)
        a[1003:b] = rng.randint(40, size=b - 1003)
        last = {}

        def fill(x):
            for k in range(b, n, D):
                m = min(D, n - k)
                x[k:k + m] = x[k - D:k - D + m]

        def f(x):
            fill(x)
            p = O.compress(2, x.tobytes(), lz_fast=True)
            hf = plen(3, x)
            last["p"] = p
            return len(p) - hf

        def ok(x):
            rest, lb = staged_checks(last["p"], n)[1]
            return rest % 32 == 0 and lb == len(last["p"])

        def move(x, p, r):
            x[p] = x[p - per] if r.rand() < 0.7 else r.randint(40)

        a, v = search(a, f, tgt, rng, lo=1003, hi=b - 8, move=move, ok=ok)
        f(a)
        if v == tgt and ok(a) and distinct3(a) == per and O.should_use(3, a.tobytes()) and O.should_use(2, a.tobytes()):
            return a
    return None


def sizes():
    """chunk sizes at the eligibility edges, short last chunks, and method subsets"""
    out = []
    for i, n in enumerate((31, 32, 99, 100, 127, 128, 129, 4096, 4097, 8191, 8192)):
        for kind in ("runs", "text", "lowcard"):
            out.append(Case("size", n, inputs.make(kind, n, 2001 + 10 * i + len(kind)), n, NATIVE, O.FIXED_MARKER))
    for i, m in enumerate((1, 3, 31, 32, 99, 100, 127, 128)):
        for chunk in (4096, 8192):
            out.append(Case("short_last", m, inputs.make("lowcard", m, 2101 + i), chunk, NATIVE, O.FIXED_MARKER))
    for ms in ((1,), (2,), (3,), (2, 3), (1, 3), (1, 2, 3)):
        for i, kind in enumerate(("runs", "text", "lowcard", "log", "skewed")):
            for n in (4096, 8192):
                out.append(Case("methods", ms, inputs.make(kind, n, 2201 + 7 * i + n), n, ms, O.FIXED_MARKER))
    return out


def match_edges():
    """Dictionary-only chunks (methods=(2,)) with beneficial payloads whose bytes (distances included) pin the match
    search: window distance 4096 / 4097, matches of 32 / 33 bytes and up to the chunk end, a 3-byte match at n - 3,
    equal-length 3-byte candidates in different fingerprint sub-buckets, overlapping sources, a bucket of > 300
    entries, and chains that never merge"""
    out = []
    rng = np.random.RandomState(2301)
    M2 = (2,)
    base = lambda n: periodic(n, 200, rng)  # noqa: E731
    for dist in (4095, 4096, 4097):
        a = base(8192)
        u = rng.randint(256, size=40).astype(np.uint8)
        a[300:340] = u
        a[300 + dist:340 + dist] = u
        out.append(Case("window", dist, a.tobytes(), 8192, M2, O.FIXED_MARKER))
    for L in (31, 32, 33, 34):
        a = base(4096)
        u = rng.randint(256, size=L).astype(np.uint8)
        a[1000:1000 + L] = u
        a[3000:3000 + L] = u
        out.append(Case("match_len", L, a.tobytes(), 4096, M2, O.FIXED_MARKER))
    for n in (4096, 8192):
        for left in (33, 32, 31, 4, 3):
            a = base(n)
            u = rng.randint(256, size=left).astype(np.uint8)
            a[500:500 + left] = u
            a[n - left:] = u  # the last token is a match that runs to the chunk's end
            out.append(Case("match_to_end", left, a.tobytes(), n, M2, O.FIXED_MARKER))
        for fourth in (0, 77):  # a 3-byte match at n - 3: the earlier trigram followed by a zero (the padding) or not
            a = base(n)
            a[700:703] = (251, 252, 253)
            a[703] = fourth
            a[n - 3:] = (251, 252, 253)
            out.append(Case("match_at_n-3", fourth, a.tobytes(), n, M2, O.FIXED_MARKER))
        # equal-length 3-byte candidates: the trigram at 2000 + 8 k followed by different bytes, the earliest wins
        a = base(n)
        for k, nxt in enumerate((11, 12, 13, 14, 15, 16, 17, 18)):
            a[2000 + 8 * k:2004 + 8 * k] = (240, 241, 242, nxt)
        a[3000:3004] = (240, 241, 242, 99)
        out.append(Case("three_byte_subbuckets", n, a.tobytes(), n, M2, O.FIXED_MARKER))
        for d in (1, 2, 3):  # overlapping sources: a period of d inside the chunk
            a = base(n)
            a[1500:1600] = np.resize(rng.randint(256, size=d).astype(np.uint8), 100)
            out.append(Case("overlap", d, a.tobytes(), n, M2, O.FIXED_MARKER))
        # a bucket of > 300 entries: "abcdefgh" + one random byte, repeated
        unit = np.frombuffer(b"abcdefgh", dtype=np.uint8)
        a = np.concatenate([np.concatenate([unit, rng.randint(256, size=1).astype(np.uint8)]) for _ in range(n // 9 + 1)])[:n]
        out.append(Case("big_bucket", n // 9, a.tobytes(), n, M2, O.FIXED_MARKER))
        # speculative chains that never merge: 37 literals, then 32-byte matches off the segment grid
        out.append(Case("no_merge", 37, periodic(n, 37, rng).tobytes(), n, M2, O.FIXED_MARKER))
    return out


def ratio_ties():
    """multi-candidate ties: (len + ovh) / size equal for two candidates (the larger keeps the tie), and one run
    (two payload bytes) either side; RLE-only chunks: 2 R1 + ovh = 2 (2 R2 + ovh)"""
    out = []
    rng = np.random.RandomState(2401)
    ovh = 18
    for cands in ((4096, 2048, 1024), (3072, 1536, 512)):  # (the library takes lists whose gcd is a multiple of 16, >= 256)
        big, half, small = cands
        R2 = 700 * half // 2048
        R3 = (R2 // 2) + 30  # the smallest candidate is clearly worse
        for d in (-1, 0, 1):
            R1 = 2 * R2 + ovh // 2 + d
            a = np.concatenate([runs_data(small, R3, rng, max_len=8), runs_data(half - small, R2 - R3, rng, max_len=8),
                                runs_data(big - half, R1 - R2, rng, max_len=8)])
            if a[small] == a[small - 1] or a[half] == a[half - 1]:
                a[small] ^= 0x80; a[half] ^= 0x80
            out.append(Case("ratio_tie", d, a.tobytes(), cands, NATIVE, O.FIXED_MARKER))
    return out


def hopeless():
    """the Dictionary trial skipped before its index when the n-gram bound reaches the cutoff (sf_lz_bound_ngrams,
    taken only when `staged` holds: a Huffman payload in hand and 100 distinct3 >= 34 min(1000, n)), cutoff =
    Huffman payload + 1: "hopeless" puts the kernel's own (hashed) bound at cutoff - 1, cutoff, cutoff + 1, which
    moves the skip; "hopeless_exact" puts the exact (4 D + 2 F) / 3 there (the hashed bound is then below it).  The
    chunks are a random prefix over 40 symbols, then copies of earlier stretches cut by a random byte, so that most
    matches end on a new 4-gram and most literals are forced: the Dictionary payload lies a few dozen bytes above
    the exact bound"""
    out = []
    rng = np.random.RandomState(2501)

    def make(n, seg, pre):
        a = np.empty(n, dtype=np.uint8)
        a[:pre] = rng.randint(40, size=pre)
        p = pre
        while p < n:
            L = min(n - p, int(rng.randint(seg - 3, seg + 4)))
            q = int(rng.randint(0, p - L))
            a[p:p + L] = a[q:q + L]
            p += L
            if p < n:
                a[p] = rng.randint(40); p += 1
        return a

    for n in (4096, 8192):
        for label, hashed in (("hopeless", True), ("hopeless_exact", False)):
            def f(x):
                hf = plen(3, x)
                if hf is None or hf + 18 >= n:
                    return None
                return ngram_bound(x, hashed) - (hf + 1)

            def ok(x):
                b = x.tobytes()
                return (O.should_use(2, b) and O.should_use(3, b) and not O.should_use(1, b)
                        and 100 * distinct3(x) >= 34 * min(1000, n))

            starts = [make(n, seg, pre) for seg in (8, 9, 10, 11, 12) for pre in (400, 600)]
            a = min((x for x in starts if f(x) is not None and ok(x)), key=lambda x: abs(f(x)))
            for tgt in (0, -1, 1):
                a, v = search(a, f, tgt, rng, lo=1003, steps=2000, ok=ok,
                              move=lambda x, p_, r: x.__setitem__(p_, x[p_ - 1 - r.randint(600)] if r.rand() < 0.5 else r.randint(40)))
                if v == tgt:
                    out.append(Case(label, v, a.tobytes(), n, NATIVE, O.FIXED_MARKER))
    return out


FAMILIES = (rle_gate, dict_gate, huff_gate, dict_huff_ties, rle_huff_ties, rle_dict_ties, rle_shortcut, benefit,
            staged, hopeless, sizes, match_edges, ratio_ties)

_CASES = []


def cases():
    """[(Case, numbers)], built once per process"""
    if not _CASES:
        for fam in FAMILIES:
            for c in fam():
                nums = numbers(c.data, c.methods, c.marker) if isinstance(c.chunk, int) else None
                _CASES.append((c, nums))
    return list(_CASES)
