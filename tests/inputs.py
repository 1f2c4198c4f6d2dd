"""Deterministic test inputs shared by the golden generator (oracle/make_golden.py),
the CPU tests and the GPU parity tests.  numpy RandomState (MT19937) streams are
stable across numpy versions, so the same name always yields the same bytes."""
import numpy as np

_WORDS = ("the quick brown fox jumps over lazy dog adaptive marker based compression chunk "
          "method huffman dictionary delta run length encoding stream header package "
          "error warning info debug request response latency status user session").split()


def _rs(seed):
    return np.random.RandomState(seed & 0x7FFFFFFF)


def text(n, seed=1):
    r = _rs(seed)
    out = bytearray()
    while len(out) < n:
        out += _WORDS[r.randint(len(_WORDS))].encode()
        out += b" " if r.randint(8) else b".\n"
    return bytes(out[:n])


def csv(n, seed=2):
    r = _rs(seed)
    out = bytearray()
    i = 0
    while len(out) < n:
        out += b"%d,%d.%03d,cat%d,2026-%02d-%02d\n" % (i + r.randint(5), r.randint(1000), r.randint(1000),
                                                      r.randint(12), 1 + r.randint(12), 1 + r.randint(28))
        i += 1
    return bytes(out[:n])


def log(n, seed=3):
    r = _rs(seed)
    lv = [b"INFO", b"WARN", b"ERROR", b"DEBUG"]
    out = bytearray()
    t = 1700000000 + r.randint(100000)
    while len(out) < n:
        t += r.randint(5)
        out += b"2026-10-18T%02d:%02d:%02d %s svc=api path=/v1/items/%d status=%d lat=%dms\n" % (
            (t // 3600) % 24, (t // 60) % 60, t % 60, lv[r.randint(4)], r.randint(500),
            (200, 200, 200, 404, 500)[r.randint(5)], r.randint(900))
    return bytes(out[:n])


def runs(n, seed=4, max_run=600):
    r = _rs(seed)
    out = bytearray()
    while len(out) < n:
        out += bytes([r.randint(256)]) * (1 + r.randint(max_run))
    return bytes(out[:n])


def lowcard(n, seed=5, k=12):
    r = _rs(seed)
    alphabet = r.choice(256, size=k, replace=False).astype(np.uint8)
    p = r.dirichlet(np.ones(k) * 0.7)
    return alphabet[r.choice(k, size=n, p=p)].tobytes()


def rand(n, seed=6):
    return _rs(seed).randint(0, 256, size=n).astype(np.uint8).tobytes()


def ramp(n, seed=7):
    return bytes((100 + i % 20) % 256 for i in range(n))


def binary_records(n, seed=8):
    """little-endian u32 counter + u16 field + 2 flag bytes: structured binary"""
    r = _rs(seed)
    m = n // 8 + 1
    rec = np.zeros((m, 8), dtype=np.uint8)
    cnt = (np.arange(m, dtype=np.uint32) * 3 + r.randint(1000)).astype("<u4")
    rec[:, 0:4] = cnt.view(np.uint8).reshape(m, 4)
    rec[:, 4:6] = r.randint(0, 40, size=(m, 2))
    rec[:, 6] = r.randint(0, 3, size=m)
    rec[:, 7] = 0
    return rec.tobytes()[:n]


def skewed(n, seed=9):
    """geometric symbol distribution: deep Huffman trees"""
    r = _rs(seed)
    v = np.minimum(r.geometric(0.5, size=n) - 1, 40).astype(np.uint8)
    return (v + 48).astype(np.uint8).tobytes()


def fib_skew(n, seed=10):
    """Fibonacci-like frequencies: maximal Huffman depth for the size"""
    f = [1, 1]
    while sum(f) + f[-1] + f[-2] <= n:
        f.append(f[-1] + f[-2])
    out = bytearray()
    for s, c in enumerate(f):
        out += bytes([65 + s]) * c
    out += bytes([65]) * (n - len(out))
    a = np.frombuffer(bytes(out), dtype=np.uint8).copy()
    _rs(seed).shuffle(a)
    return a.tobytes()


def periodic(n, seed=11, period=45):
    base = rand(period, seed)
    return (base * (n // period + 1))[:n]


def ties(n, seed=12):
    """many equal frequencies: exercises the (weight, leader) tie-break"""
    k = 1 + _rs(seed).randint(2, 200)
    a = np.arange(n, dtype=np.int64) % k
    a = (a * 7 + 3) % 256
    return a.astype(np.uint8).tobytes()


KINDS = {"text": text, "csv": csv, "log": log, "runs": runs, "lowcard": lowcard, "rand": rand, "ramp": ramp,
         "binrec": binary_records, "skewed": skewed, "fib": fib_skew, "periodic": periodic, "ties": ties}


def make(kind, n, seed):
    return KINDS[kind](n, seed)


# ---- the named inputs of SURVEY.md §8(c) (recur in the reference's own tests) ----
def survey_inputs():
    A = b"AAAABBBCCDAAAABBBCCDA" * 20                       # compression_methods.py:719
    B = bytes((i * i) % 17 + 65 for i in range(4096))
    C = (b"The quick brown fox jumps over the lazy dog. " * 100)[:4096]
    D = b"A" * 1000 + b"B" * 1000 + b"C" * 1000               # tests/test_compression.py:27
    E = bytes((100 + i % 20) % 256 for i in range(1000))      # test_basic_compression.py:38-40
    F = bytes((i * 167 + 13) % 256 for i in range(4096))
    G = b"".join(b"%d,%d.%03d,row%d\n" % (i, (i * 37) % 1000, (i * 91) % 1000, i % 7) for i in range(400))[:4096]
    T = b"This is a test text file with some repeating content. " * 30  # tests/test_compression.py:39
    return {"A": A, "B": B, "C": C, "D": D, "E": E, "F": F, "G": G, "T": T}


def codec_cases():
    """(name, bytes) for per-codec known-answer tests"""
    cases = list(survey_inputs().items())
    spec = [("text", 4096), ("text", 1000), ("csv", 4096), ("csv", 2048), ("log", 4096), ("log", 8192),
            ("runs", 4096), ("runs", 3000), ("runs", 700), ("lowcard", 4096), ("lowcard", 512), ("rand", 4096),
            ("rand", 300), ("ramp", 4096), ("binrec", 4096), ("binrec", 8192), ("skewed", 4096), ("fib", 4096),
            ("fib", 8192), ("periodic", 4096), ("ties", 4096), ("ties", 1024), ("text", 8192), ("text", 129),
            ("text", 100), ("text", 99), ("text", 33), ("text", 32), ("text", 31), ("text", 5), ("text", 4),
            ("text", 3), ("text", 2), ("text", 1), ("runs", 1024), ("lowcard", 1023), ("csv", 1003), ("csv", 1002)]
    for i, (k, n) in enumerate(spec):
        cases.append(("%s_%d_s%d" % (k, n, 100 + i), make(k, n, 100 + i)))
    cases.append(("zeros_4096", bytes(4096)))
    cases.append(("one_sym_300", b"z" * 300))
    cases.append(("two_sym_4096", (b"ab" * 2048)))
    cases.append(("all256_4096", bytes(range(256)) * 16))
    cases.append(("run256_then_text", b"Q" * 256 + text(3840, 77)))
    cases.append(("run255x3", b"Q" * 765 + b"R" * 255 + b"S" * 254 + b"T"))
    cases.append(("empty", b""))
    return cases


def mixed_file(n_chunks, chunk, seed, kinds=("text", "csv", "log", "runs", "lowcard", "binrec", "periodic")):
    r = _rs(seed)
    parts = []
    for i in range(n_chunks):
        k = kinds[r.randint(len(kinds))]
        parts.append(make(k, chunk, seed * 1000 + i))
    return b"".join(parts)


def container_cases():
    """(name, data, cfg) for whole-.ambc known-answer tests; cfg keys as ref_harness.make_compressor"""
    S = survey_inputs()
    out = []
    out.append(("H1", S["C"] + S["D"] + S["B"] + S["G"] + S["A"], dict(chunk_size=4096)))
    out.append(("H2", S["C"] + S["F"] + S["C"] + S["D"], dict(chunk_size=4096)))
    tail = text(4096, 31) + runs(4096, 32) + text(4096, 33) + rand(4096, 34) + text(4096, 35) + runs(1000, 36)
    out.append(("tailraw", tail, dict(chunk_size=4096)))
    out.append(("tailraw_pcr", tail, dict(chunk_size=4096, per_chunk_raw=True)))
    out.append(("mixed12_4096", mixed_file(12, 4096, 41) + text(777, 42), dict(chunk_size=4096)))
    out.append(("mixed16_1024", mixed_file(16, 1024, 43) + csv(100, 44), dict(chunk_size=1024)))
    out.append(("mixed8_2048", mixed_file(8, 2048, 45) + runs(31, 46), dict(chunk_size=2048)))
    out.append(("mixed4_8192", mixed_file(4, 8192, 47, ("text", "log", "csv", "lowcard")), dict(chunk_size=8192)))
    out.append(("mixed10_512", mixed_file(10, 512, 48) + lowcard(40, 49), dict(chunk_size=512)))
    out.append(("mixed6_3000", mixed_file(6, 3000, 50), dict(chunk_size=3000)))
    out.append(("c16384_degenerate", mixed_file(3, 16384, 51, ("text", "log")), dict(chunk_size=16384)))
    out.append(("only_rle", mixed_file(6, 4096, 52), dict(chunk_size=4096, method_ids=(1,))))
    out.append(("only_huff", mixed_file(6, 4096, 53, ("csv", "lowcard", "skewed", "text")), dict(chunk_size=4096, method_ids=(3,))))
    out.append(("only_dict_delta", mixed_file(5, 4096, 54), dict(chunk_size=4096, method_ids=(2, 4))))
    out.append(("rle_huff", mixed_file(8, 4096, 55), dict(chunk_size=4096, method_ids=(1, 3))))
    out.append(("random_verbatim", rand(6000, 56), dict(chunk_size=4096)))
    out.append(("tiny_31", text(31, 57), dict(chunk_size=4096)))
    out.append(("tiny_200", text(200, 58), dict(chunk_size=4096)))
    out.append(("empty", b"", dict(chunk_size=4096)))
    out.append(("short_last", mixed_file(3, 4096, 59) + text(20, 60), dict(chunk_size=4096)))
    out.append(("repeated_abc", S["D"], dict(chunk_size=4096)))   # tests/test_compression.py:27
    out.append(("text_T", S["T"], dict(chunk_size=4096)))        # tests/test_compression.py:39
    out.append(("found_marker", mixed_file(5, 4096, 61) + text(300, 62), dict(chunk_size=4096, found_marker=True)))
    return out


REF_DEFAULT_CANDIDATES = (131072, 65536, 32768, 16384, 8192, 4096, 2048, 1024)  # adaptive_compressor.py:61-62


def dynamic_cases():
    """(name, data, cfg) for the reference's multi-candidate mode (adaptive_compressor.py:548-584):
    every candidate size is tried at every position, the best ratio wins, larger sizes win ties"""
    out = []
    out.append(("dyn_default_mixed", mixed_file(9, 4096, 71, ("text", "csv", "log", "runs", "lowcard")) + text(700, 72),
                dict(chunk_size=REF_DEFAULT_CANDIDATES)))
    out.append(("dyn_default_tailraw", text(4096, 73) + runs(3000, 74) + csv(5000, 75) + rand(3000, 76) + text(500, 77),
                dict(chunk_size=REF_DEFAULT_CANDIDATES)))
    out.append(("dyn_small", mixed_file(10, 1024, 78) + lowcard(300, 79), dict(chunk_size=(2048, 1024, 512))))
    out.append(("dyn_no8192", mixed_file(5, 4096, 80, ("text", "log", "csv")) + log(2500, 81),
                dict(chunk_size=(16384, 4096, 1024))))
    out.append(("dyn_rle_huff", mixed_file(6, 2048, 82, ("runs", "lowcard", "skewed")), dict(chunk_size=(4096, 2048, 1024), method_ids=(1, 3))))
    return out


def marker_cases():
    """(name, data, max_len, sample_size)"""
    return [
        ("abc100", b"ABC" * 100, 16, None),               # tests/test_marker_finder.py:21
        ("a1000", b"A" * 1000, 24, None),                 # :61
        ("ab500", b"AB" * 500, 24, None),                 # :62
        ("all256x4", bytes(range(256)) * 4, 24, None),    # :63
        ("rand1000", rand(1000, 71), 16, None),
        ("rand2000", rand(2000, 72), 24, None),
        ("rand4096", rand(4096, 73), 32, None),
        ("text3000", text(3000, 74), 32, None),
        ("log3000", log(3000, 75), 32, None),
        ("sample", rand(10000, 76), 16, 1000),            # :44-56 (sampling branch)
        ("sample_text", text(20000, 77), 32, 1500),
        ("empty", b"", 8, None),
        ("one", b"\x00", 8, None),
        ("ff", b"\xff" * 64, 8, None),
        ("limit_fail", rand(4096, 78), 8, None),          # ValueError: nothing absent up to 8 bits
    ]


def malformed_payloads():
    """(name, method id, payload bytes, orig_len) -- decoder edge cases (SURVEY.md §3.3)"""
    S = survey_inputs()
    out = []
    out.append(("rle_empty", 1, b"", 10))
    out.append(("rle_odd", 1, b"A\x03B\x02C", 5))
    out.append(("rle_short", 1, b"A\x03", 10))
    out.append(("rle_long", 1, b"A\xffB\xff", 100))
    out.append(("rle_zero_count", 1, b"A\x00B\x02", 2))
    out.append(("lz_empty", 2, b"", 10))
    out.append(("lz_lit_trunc", 2, b"\x00A\x00", 5))
    out.append(("lz_match_trunc", 2, b"\x00A\x01\x01\x00", 5))
    out.append(("lz_dist0", 2, b"\x00A\x01\x00\x00\x05", 6))
    out.append(("lz_dist0_empty", 2, b"\x01\x00\x00\x05\x00", 6))
    out.append(("lz_overlap", 2, b"\x00A\x00B\x01\x02\x00\x09", 11))
    out.append(("lz_neg_index", 2, b"\x00A\x00B\x00C\x01\x05\x00\x04\x00Z", 9))
    out.append(("lz_neg_index_err", 2, b"\x00A\x01\x09\x00\x04\x00Z", 9))
    out.append(("lz_flag7", 2, b"\x00A\x07\x01\x00\x03\x00B", 6))
    out.append(("lz_short_out", 2, b"\x00A\x00B", 10))
    out.append(("lz_long_match", 2, b"\x00A\x01\x01\x00\xff", 20))
    out.append(("huff_empty", 3, b"", 10))
    out.append(("huff_k0", 3, b"\x00\x00\x00\x00\x00", 4))
    out.append(("huff_k1", 3, b"\x01A\x05\x00\x00\x00\x05\x00\x00\x00\x00", 5))
    out.append(("huff_trunc_table", 3, b"\x03A\x05\x00\x00\x00B", 5))
    out.append(("delta_empty", 4, b"", 4))
    out.append(("delta_short", 4, b"\x05\x01\x01", 6))
    out.append(("delta_long", 4, b"\x05\x01\x01\xff\xff", 3))
    out.append(("raw_short", 255, b"abc", 6))
    out.append(("raw_long", 255, b"abcdef", 3))
    return out


def corrupt(payload, r):
    """1 to 3 random edits of a payload drawn from RandomState r: a byte overwritten, the tail cut off, or a few
    random bytes appended"""
    a = bytearray(payload)
    for _ in range(int(r.randint(1, 4))):
        what = r.randint(3)
        if what == 0 and len(a) > 2:
            a[r.randint(len(a))] = r.randint(256)
        elif what == 1 and len(a) > 4:
            del a[r.randint(len(a)):]
        else:
            a += bytes(r.randint(0, 256, size=r.randint(1, 5)).astype(np.uint8))
    return bytes(a)


def gate_case(i):
    """i-th should_use probe: a seeded input blended with random bytes so that the
    sampled ratios / entropy land near the reference's thresholds."""
    kinds = sorted(KINDS)
    r = _rs(900000 + i)
    k = kinds[r.randint(len(kinds))]
    n = int(r.choice([3, 4, 31, 99, 100, 101, 500, 999, 1000, 1001, 1003, 1500, 2048, 4096, 5000, 8192]))
    frac = float(r.choice([0.0, 0.0, 0.2, 0.5, 0.7, 0.9]))
    data = make(k, n, 5000 + i)
    if frac and n > 8:
        a = np.frombuffer(data, dtype=np.uint8).copy()
        m = r.rand(n) < frac
        a[m] = r.randint(0, 256, size=int(m.sum()))
        data = a.tobytes()
    return k, n, frac, data


N_GATE_CASES = 400
