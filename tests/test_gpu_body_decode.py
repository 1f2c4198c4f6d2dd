"""Body decode (ambc_decompress_dev) against an expected-output model built from the oracle codecs, on every
decode kernel's own path: well-formed and malformed packages in every dispatch class of ambc_decode_launch,
destinations at every residue mod 16, neighbouring packages of different kernels, tables long enough for a
second round of every kernel's table loop, and a body and output past 2^32 bytes.

The model (CPU, no library): walk the body as the reference does (adaptive_compressor.py:396-454), decode each
package's payload with the oracle, and place it at the output offset the index gives it, which is the sum of
the nominal lengths before it (decode.cu: nominal_out).  Where the reference's codec raises, the slice is
zeros and status[0] counts it (:440-442); where the decoded length differs from the nominal length, the slice
is the decoded bytes cut or zero padded to its length and status[1] counts it (include/ambc.h); the output
behind the last package is zeros up to orig_size (:447-452)."""
import numpy as np
import pytest

import inputs
import oracle as O

MARKER = O.FIXED_MARKER
HDR = len(MARKER) + 14
KNOWN = (1, 2, 3, 4, 255)
UNKNOWN = 77          # a type no decoder knows: its payload is copied through (:432-435)
GUARD = 64            # bytes behind orig_size that the decode must not touch
FILL = 0xA5           # what the output holds before the decode: every byte the decode owes is checked

# first-round sizes of the table loops (decode.cu: ambc_decode_launch): grid x entries looked at per round
ROUND_WARP = 148 * 16 * 8 * 64      # k_decode_warp: 18,944 CTAs x 64 lanes
ROUND_LZ = 148 * 24 * 8 * 32        # k_decode_lz: 3,552 CTAs x 8 warps x 32 lanes
ROUND_CTA = 148 * 6 * 256           # k_decode: 888 CTAs x 256 threads


def header(t, orig, comp):
    return MARKER + bytes([t, 0]) + int(orig).to_bytes(4, "little") * 2 + int(comp).to_bytes(4, "little")


def nominal(t, comp, orig):
    """bytes the reference appends for a package, knowable without decoding (decode.cu: nominal_out)"""
    if t not in KNOWN:
        return comp
    if t == 255:
        return orig
    if comp == 0:
        return 0
    return min(comp, orig) if t == 4 else orig


def kernel_class(t, comp, orig):
    """the decoder ambc_decode_launch gives a table entry (raw pieces and unknown types are entries of type 255)"""
    if t == 255:
        return "raw"
    if t in (1, 3) and comp <= 8192 and orig <= 8192:
        return "warp4096" if comp <= 4096 and orig <= 4096 else "warp8192"
    if t == 2 and comp <= 8192 and orig <= 8192:
        return "lz4096" if orig <= 4096 else "lz8192"
    if t == 4 and comp <= 8192 and orig <= 8192:
        return "cta_fast"
    return "cta_serial"


CLASS_TYPES = {"warp4096": (1, 3), "warp8192": (1, 3), "lz4096": (2,), "lz8192": (2,), "cta_fast": (4,),
               "cta_serial": (1, 2, 3, 4), "raw": (255,)}
# the decoders of these types return the nominal length for every payload (RLE pads / truncates to orig_len,
# Delta returns min(comp_len, orig_len), raw pads / truncates): their packages never raise or mismatch
NEVER_BAD = (1, 4, 255)


def model(body, orig_size, marker=MARKER):
    """-> (expected output bytes, expected status [raised, mismatched], packages).  A package is a dict of the
    header fields, its payload offset, dst_off, out_len and outcome ('clean' / 'raise' / 'mismatch'); packages
    that own no output bytes are listed with out_len 0 and decoded by nobody."""
    body = bytes(body)
    mb = len(marker)
    hdr = mb + 14
    out = bytearray(orig_size)
    status = [0, 0]
    pkgs = []
    pos = o = 0
    while pos < len(body):
        if pos + hdr > len(body):
            break
        if body[pos:pos + mb] != marker:
            raise ValueError("Marker mismatch in chunk header.")
        t = body[pos + mb]
        orig = int.from_bytes(body[pos + mb + 6:pos + mb + 10], "little")
        comp = int.from_bytes(body[pos + mb + 10:pos + mb + 14], "little")
        pos += hdr
        if t == 0 or pos + comp > len(body):
            break
        p = body[pos:pos + comp]
        nom = nominal(t, comp, orig)
        out_len = max(0, min(nom, orig_size - o))
        rec = dict(type=t, orig=orig, comp=comp, src=pos, dst=o, out_len=out_len, outcome="clean")
        if out_len:
            w = O.decompress(t, p, orig) if t in KNOWN else p
            if isinstance(w, int):
                rec["outcome"] = "raise"
                status[0] += 1
            else:
                out[o:o + out_len] = (w + bytes(max(0, out_len - len(w))))[:out_len]
                if len(w) != nom:
                    rec["outcome"] = "mismatch"
                    status[1] += 1
        pkgs.append(rec)
        pos += comp
        o += nom
        if o >= orig_size:  # :444-445
            break
    return bytes(out), status, pkgs


# ---- bodies ------------------------------------------------------------------------------------------------
class BodyBuilder:
    """packages appended one by one; tracks the output offset so that a raw pad can put the next package's
    destination at a chosen residue mod 16"""

    def __init__(self):
        self.parts = []
        self.len = 0
        self.out = 0
        self.tags = {}   # payload offset -> where the payload came from

    def add(self, t, orig, payload, tag="valid"):
        self.parts.append(header(t, orig, len(payload)))
        self.parts.append(payload)
        self.tags[self.len + HDR] = tag
        self.len += HDR + len(payload)
        self.out += nominal(t, len(payload), orig)

    def pad_to(self, residue, r):
        k = (residue - self.out) % 16
        if k:
            self.add(255, k, bytes(r.randint(0, 256, size=k).astype(np.uint8)), "pad")

    def bytes(self):
        return b"".join(self.parts)


def _junk(r, n):
    return bytes(r.randint(0, 256, size=max(n, 0)).astype(np.uint8))


def place(cls, t, p, o, r):
    """(payload, orig_len) that put package (t, p, o) into decoder class cls, by choosing orig_len and appending
    trailing bytes (the oracle defines what they mean), or None where the payload is too long for the class"""
    if not p:
        return None
    if cls == "cta_serial":
        if len(p) > 8192 or o > 8192:
            return p, o
        if r.randint(2):
            return p + _junk(r, 8193 - len(p) + r.randint(0, 3000)), o
        return p, 8193 + r.randint(0, 12000)
    cmax, omin, omax = {"warp4096": (4096, 1, 4096), "warp8192": (8192, 1, 8192), "lz4096": (8192, 1, 4096),
                        "lz8192": (8192, 4097, 8192), "cta_fast": (8192, 1, 8192)}[cls]
    if len(p) > cmax:
        return None
    if not omin <= o <= omax:
        o = int(r.randint(omin, omax + 1))
    if cls == "warp8192" and len(p) <= 4096 and o <= 4096:
        if r.randint(2):
            p = p + _junk(r, int(r.randint(4097, 8193)) - len(p))
        else:
            o = int(r.randint(4097, 8193))
    elif r.randint(4) == 0:
        p = p + _junk(r, int(r.randint(len(p), cmax + 1)) - len(p))
    return p, o


TYPE_CLASSES = {1: ("warp4096", "warp8192", "cta_serial"), 3: ("warp4096", "warp8192", "cta_serial"),
                2: ("lz4096", "lz8192", "cta_serial"), 4: ("cta_fast", "cta_serial")}


def dispatch_sources():
    """(type, payload, orig_len, tag): the golden decode vectors of the reference, corrupted oracle payloads
    (the generator of test_decode_corrupted_fuzz) and valid oracle payloads around the class limits"""
    import json
    import os
    g = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "decode_kat.json")))
    src = [(row["method"], bytes.fromhex(row["payload"]), row["orig_len"], "golden") for row in g]
    r = np.random.RandomState(77)
    kinds = sorted(inputs.KINDS)
    for mid in (1, 2, 3, 4):
        for i in range(60):
            d = inputs.make(kinds[r.randint(len(kinds))], int(r.choice([64, 300, 1024, 4096])), 40000 + i)
            p = O.compress(mid, d, lz_fast=True)
            if not isinstance(p, int):
                src.append((mid, inputs.corrupt(p, r), len(d), "malformed"))
    for n in (4096, 4097, 8192, 8193, 20000):
        for j, kind in enumerate(("text", "runs", "lowcard", "skewed", "binrec", "rand")):
            d = inputs.make(kind, n, 61000 + 10 * n + j)
            for mid in (1, 2, 3, 4):
                p = O.compress(mid, d, lz_fast=True)
                if not isinstance(p, int):
                    src.append((mid, p, n, "valid"))
    return src


def dispatch_cases(seed):
    """(type, orig_len, payload, tag, class) covering every decoder class, shuffled so that the classes
    interleave"""
    r = np.random.RandomState(seed)
    cases = []
    for t, p, o, tag in dispatch_sources():
        if t == 255:
            cases.append((255, o, p, tag, "raw"))
            continue
        for cls in TYPE_CLASSES[t]:
            pl = place(cls, t, p, o, r)
            if pl is not None:
                assert kernel_class(t, len(pl[0]), pl[1]) == cls, (t, len(pl[0]), pl[1], cls)
                cases.append((t, pl[1], pl[0], tag, cls))
    # raw packages: padded, truncated, across 64 KiB pieces; unknown types are copied through as raw pieces
    for n in (1, 7, 300, 4095, 4097, 8193, 65535, 65536, 65537, 70001, 131073, 200003):
        for comp in (n, max(1, n - 1 - int(r.randint(0, n))), n + 1 + int(r.randint(0, 5000))):
            cases.append((255, n, _junk(r, comp), "valid", "raw"))
    for comp in (1, 100, 4097, 65537, 70001):
        cases.append((UNKNOWN, 1 + int(r.randint(0, 9000)), _junk(r, comp), "valid", "raw"))
    order = r.permutation(len(cases))
    return [cases[i] for i in order]


def build_body(cases, seed, pads=True, tail=1000):
    """-> (body, orig_size, tags).  With pads, a raw package of 0..15 bytes in front of each case walks the
    destinations of every class through all 16 residues mod 16."""
    r = np.random.RandomState(seed)
    b = BodyBuilder()
    seen = {}
    for t, o, p, tag, cls in cases:
        if pads:
            k = seen.get(cls, 0)
            seen[cls] = k + 1
            b.pad_to(k % 16, r)
        b.add(t, o, p, tag)
    return b.bytes(), b.out + tail, b.tags


# ---- coverage ------------------------------------------------------------------------------------------------
def entry_classes(table):
    return [kernel_class(int(e["type"]), int(e["comp_len"]), int(e["orig_len"])) for e in table]


def check_matrix_coverage(table, pkgs, tags):
    """every (class x type) cell holds clean packages and packages that raise or mismatch (malformed payloads
    where the type's decoder never does), every class sees all 16 destination residues"""
    cls = entry_classes(table)
    for c, types in CLASS_TYPES.items():
        res = {int(e["dst_off"]) % 16 for e, k in zip(table, cls) if k == c}
        assert res == set(range(16)), (c, sorted(res))
    cells = {}
    for p in pkgs:
        if not p["out_len"]:
            continue
        t = p["type"] if p["type"] in KNOWN else 255
        c = kernel_class(t, p["comp"], p["orig"])
        cells.setdefault((c, t), set()).update({p["outcome"], tags.get(p["src"], "valid")})
    for c, types in CLASS_TYPES.items():
        for t in types:
            got = cells.get((c, t), set())
            assert "clean" in got, (c, t, got)
            if t in NEVER_BAD:
                assert "malformed" in got or "golden" in got, (c, t, got)
            else:
                assert "raise" in got and "mismatch" in got, (c, t, got)


# ---- CPU: the model against the reference's own body decode ------------------------------------------------------
def _container_bodies():
    for name, data, cfg in inputs.container_cases():
        marker = MARKER
        if cfg.get("found_marker"):
            marker = O.marker_aligned(*O.find_marker(data, 32))
        body, _ = O.compress_body(data, cfg["chunk_size"], tuple(cfg.get("method_ids", (1, 2, 3, 4))), marker,
                                  bool(cfg.get("per_chunk_raw")))
        yield name, body, len(data), marker, data


def test_model_equals_reference_on_container_bodies():
    """oracle-compressed bodies of every container case, decoded to their own length, shorter and longer: the
    model reports [0, 0] and equals the reference's body decode"""
    for name, body, n, marker, data in _container_bodies():
        for size in (n, n // 2, max(n - 1, 0), n + 777):
            out, status, _ = model(body, size, marker)
            assert status == [0, 0], (name, size)
            assert out == O.decompress_body(body, size, marker), (name, size)
        assert model(body, n, marker)[0] == data, name


def test_model_equals_reference_on_hand_built_bodies():
    """hand-built bodies: raw packages padded and truncated, unknown types, an END package, a payload cut off
    by the body's end, orig_size cutting a package: where the model reports [0, 0] it equals the reference"""
    r = np.random.RandomState(5)
    d = inputs.text(5000, 9)
    parts = [header(1, 5000, 0) + b"",
             header(2, 5000, len(O.compress(2, d))) + O.compress(2, d),
             header(255, 70000, 3) + b"abc",
             header(255, 10, 20) + _junk(r, 20),
             header(UNKNOWN, 99, 65537) + _junk(r, 65537),
             header(3, 3000, len(O.compress(3, d[:3000]))) + O.compress(3, d[:3000]),
             header(4, 7000, 5000) + O.compress(4, d),
             header(1, 4000, len(O.compress(1, d[:4000]))) + O.compress(1, d[:4000])]
    full = b"".join(parts)
    total = sum(nominal(t, c, o) for t, o, c in [(1, 5000, 0), (2, 5000, 1), (255, 70000, 3), (255, 10, 20),
                                                 (UNKNOWN, 99, 65537), (3, 3000, 1), (4, 7000, 5000), (1, 4000, 1)])
    bodies = [full, full + header(0, 0, 0) + parts[1], full[:-7], full + header(2, 10, 1 << 20) + b"xyz"]
    for body in bodies:
        for size in (0, 1, 5000, 5001, 75009, total - 1, total, total + 4096):
            out, status, pkgs = model(body, size)
            assert status == [0, 0], size
            assert out == O.decompress_body(body, size), size
    out, _, pkgs = model(full, total)
    assert [p["dst"] for p in pkgs if p["out_len"]] == [0, 5000, 75000, 75010, 140547, 143547, 148547]


def test_model_walk_equals_host_index():
    """the model's walk places every package where ambc_index_host does (raw packages as pieces of 64 KiB)"""
    from adaptive_compression_b200 import engine
    cases = dispatch_cases(11)
    body, size, _ = build_body(cases[:400], 12)
    _, _, pkgs = model(body, size)
    table, covered = engine.index_host(np.frombuffer(body, dtype=np.uint8), size)
    want = []
    for p in pkgs:
        if not p["out_len"]:
            continue
        if p["type"] in (1, 2, 3, 4):
            want.append((p["type"], p["src"], p["dst"], p["comp"], p["orig"], p["out_len"]))
            continue
        for k in range(0, p["out_len"], 65536):
            piece = min(65536, p["out_len"] - k)
            want.append((255, p["src"] + k, p["dst"] + k, max(0, min(p["comp"] - k, piece)), piece, piece))
    got = [(int(e["type"]), int(e["src_off"]), int(e["dst_off"]), int(e["comp_len"]), int(e["orig_len"]),
            int(e["out_len"])) for e in table]
    assert got == want
    assert covered == sum(p["out_len"] for p in pkgs)


def test_model_slices_equal_golden_decode_vectors(golden):
    """a golden vector alone in a body: the model's slice is the reference's output, and the status names what
    the reference did (raised / returned another length than the nominal one)"""
    for row in golden["decode_kat"]:
        t, p, o = row["method"], bytes.fromhex(row["payload"]), row["orig_len"]
        nom = nominal(t, len(p), o)
        out, status, _ = model(header(t, o, len(p)) + p, nom)
        if row["error"]:
            assert out == bytes(nom) and status == [1, 0], row["name"]
        else:
            want = bytes.fromhex(row["out"])
            assert out == (want + bytes(nom))[:nom], row["name"]
            assert status == [0, int(len(want) != nom and nom > 0)], row["name"]


def test_dispatch_matrix_coverage():
    """the body of test_dispatch_matrix, from its host index table: every (class x type) cell holds clean
    packages and failing ones (malformed payloads for RLE, Delta and raw), every class all 16 residues"""
    from adaptive_compression_b200 import engine
    body, size, tags = build_body(dispatch_cases(21), 22)
    _, _, pkgs = model(body, size)
    table, _ = engine.index_host(np.frombuffer(body, dtype=np.uint8), size)
    check_matrix_coverage(table, pkgs, tags)


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    from adaptive_compression_b200 import engine
    engine.require_cuda()
    return engine


def _prefilled(n):
    import torch
    return torch.full((n + GUARD,), FILL, dtype=torch.uint8, device="cuda")


def _diff_report(got, want, pkgs):
    """-> (differing bytes, [(type, class, dst_off, out_len, outcome, first differing byte in the slice, count)])"""
    bad = np.flatnonzero(got != want)
    rep = []
    for p in pkgs:
        if p["out_len"] and len(rep) < 12:
            lo, hi = np.searchsorted(bad, [p["dst"], p["dst"] + p["out_len"]])
            if hi > lo:
                rep.append((p["type"], kernel_class(p["type"] if p["type"] in KNOWN else 255, p["comp"], p["orig"]),
                            p["dst"], p["out_len"], p["outcome"], int(bad[lo]) - p["dst"], int(hi - lo)))
    return len(bad), rep


def _decode_and_check(eng, body, size, gpu_index):
    import torch
    want, want_status, pkgs = model(body, size)
    t_body = torch.frombuffer(bytearray(body), dtype=torch.uint8).cuda()
    out = _prefilled(size)
    _, status = eng.decompress_device(t_body, size, out=out, gpu_index=gpu_index,
                                        body_host=None if gpu_index else np.frombuffer(body, dtype=np.uint8))
    got = out.cpu().numpy()
    assert (got[size:] == FILL).all(), "bytes behind orig_size were written"
    w = np.frombuffer(want, dtype=np.uint8)
    if not np.array_equal(got[:size], w):
        pytest.fail("output differs from the model: %d bytes, packages %s" % _diff_report(got[:size], w, pkgs))
    assert status == want_status
    return pkgs


@pytest.mark.gpu
@pytest.mark.parametrize("gpu_index", [True, False])
def test_dispatch_matrix(eng, gpu_index):
    """every decoder class x type, clean / raising / mismatching / malformed payloads, destinations at every
    residue mod 16: output (zero fill and zero tail included) and status equal the model, through the device
    index and through the host index"""
    body, size, _ = build_body(dispatch_cases(21), 22)  # (its coverage: test_dispatch_matrix_coverage)
    _decode_and_check(eng, body, size, gpu_index)


@pytest.mark.gpu
def test_neighbours(eng):
    """no pads: packages of different decoders back to back at odd destinations, decoded by kernels that run
    at the same time (k_decode_lz on its side stream); a store past out_len shows in the next slice"""
    by_cls = {}
    for c in dispatch_cases(31):
        by_cls.setdefault(c[4], []).append(c)
    inter = [v[k] for k in range(40) for _, v in sorted(by_cls.items())]
    body, size, _ = build_body(inter, 32, pads=False, tail=0)
    pkgs = _decode_and_check(eng, body, size, True)
    owned = [p for p in pkgs if p["out_len"]]
    kinds = [kernel_class(p["type"] if p["type"] in KNOWN else 255, p["comp"], p["orig"]) for p in owned]
    assert sum(a != b for a, b in zip(kinds, kinds[1:])) > 0.9 * len(kinds)
    assert len({p["dst"] % 16 for p in owned}) == 16


@pytest.mark.gpu
def test_empty_payload_entries(eng):
    """table entries of a caller that own no output bytes (comp_len 0, out_len 0), in every decoder class:
    nothing is written for them and they count as neither error nor mismatch (an empty payload decodes to
    b'', its nominal length)"""
    import torch
    cases = dispatch_cases(41)[:200]
    body, size, _ = build_body(cases, 42)
    want, want_status, _ = model(body, size)
    table, _ = eng.index_host(np.frombuffer(body, dtype=np.uint8), size)
    extra = [(t, o) for t in (1, 2, 3, 4) for o in (100, 5000, 9000)] * 4
    assert {kernel_class(t, 0, o) for t, o in extra} == set(CLASS_TYPES) - {"raw"}
    rows = []
    for i, e in enumerate(table):
        rows.append(e)
        if i % 5 == 2 and extra and i + 1 < len(table):  # (the last entry stays last: the zero tail starts behind it)
            t, o = extra.pop()
            x = e.copy()
            x["comp_len"], x["orig_len"], x["type"], x["out_len"] = 0, o, t, 0
            rows.append(x)
    assert not extra
    mixed = np.array(rows, dtype=table.dtype)
    t_body = torch.frombuffer(bytearray(body), dtype=torch.uint8).cuda()
    t_table = torch.from_numpy(mixed.view(np.uint8).reshape(-1).copy()).cuda()
    out = _prefilled(size)
    _, status = eng.range_decode(t_body, t_table, len(mixed), size, out=out)
    got = out.cpu().numpy()
    assert (got[size:] == FILL).all()
    assert bytes(got[:size]) == want
    assert status == want_status


def _tile_check(out, unit_out, reps, rows=256):
    """out[:reps * len(unit_out)] == unit_out repeated, compared on the device in blocks of `rows` units"""
    import torch
    u = unit_out.numel()
    v = out[:reps * u].view(reps, u)
    for r0 in range(0, reps, rows):
        r1 = min(reps, r0 + rows)
        blk = v[r0:r1]
        if not torch.equal(blk, unit_out.expand(r1 - r0, u)):
            bad = (blk != unit_out).nonzero()[:5].tolist()
            pytest.fail("unit copies %d..%d differ from the model: (copy, byte) %s" % (r0, r1, bad))


def _small_unit(seed):
    """a few hundred distinct packages of types 1, 2 and 3 with outputs of 32..200 bytes (some malformed) and
    Delta packages, in interleaved order"""
    r = np.random.RandomState(seed)
    kinds = sorted(inputs.KINDS)
    b = BodyBuilder()
    for i in range(363):
        n = int(r.randint(32, 201))
        d = inputs.make(kinds[r.randint(len(kinds))], n, 90000 + i)
        t = (1, 2, 3, 4, 1, 2, 3, 4, 1, 2, 3)[i % 11]
        p = O.compress(t, d, lz_fast=True)
        if isinstance(p, int):  # (a Huffman table of one symbol)
            t, p = 1, O.compress(1, d)
        if i % 5 == 0:
            p = inputs.corrupt(p, r)
        b.add(t, n if r.randint(6) else int(np.clip(n + r.randint(-20, 21), 32, 200)), p)
    return b.bytes(), b.out


@pytest.mark.gpu
@pytest.mark.parametrize("gpu_index", [True, False])
def test_table_loop_second_rounds(eng, gpu_index):
    """a body of 1.3 M+ small packages of types 1, 2, 3 and 230 k+ Delta packages, tiled on the device: every
    decoder's table loop runs a second round (past 18,944 x 64, 3,552 x 8 x 32 and 888 x 256 entries), output
    and status equal the tiled model"""
    import torch
    unit, unit_size = _small_unit(51)
    want, st, pkgs = model(unit, unit_size)
    n_small = sum(p["type"] != 4 for p in pkgs if p["out_len"])  # (a corrupted payload may have become empty)
    n_delta = sum(p["type"] == 4 for p in pkgs if p["out_len"])
    reps = max(-(-1_300_000 // n_small), -(-230_000 // n_delta))
    t_unit = torch.frombuffer(bytearray(unit), dtype=torch.uint8).cuda()
    t_body = t_unit.repeat(reps)
    size = unit_size * reps
    out = _prefilled(size)
    body_host = None if gpu_index else t_body.cpu().numpy()
    _, status = eng.decompress_device(t_body, size, out=out, gpu_index=gpu_index, body_host=body_host)
    assert status == [st[0] * reps, st[1] * reps], (status, st, reps)
    assert st[0] and st[1]
    _tile_check(out, torch.frombuffer(bytearray(want), dtype=torch.uint8).cuda(), reps)
    assert (out[size:] == FILL).all()
    if gpu_index:
        tab = _device_table(eng, t_body, size)
        m = len(tab) // reps
        assert m * reps == len(tab)
        cls = np.array(entry_classes(tab[:m]) * reps)
        assert (cls[ROUND_WARP:] == "warp4096").any() and (cls[ROUND_LZ:] == "lz4096").any() \
            and (cls[ROUND_CTA:] == "cta_fast").any()
        assert int((cls != "cta_fast").sum()) >= 1_300_000 and int((cls == "cta_fast").sum()) >= 230_000


def _device_table(eng, t_body, size):
    """ambc_index_dev's table as a host array of ambc_pkg"""
    t_table, n, covered = eng.index_device(t_body, size)
    assert covered == size
    dt = np.dtype([("src_off", "<u8"), ("dst_off", "<u8"), ("comp_len", "<u4"), ("orig_len", "<u4"),
                   ("type", "<u4"), ("out_len", "<u4")])
    return t_table[:n * 32].cpu().numpy().view(dt)


def _big_unit(seed):
    """~1 MiB of packages from every class, raw-heavy (raw packages across 64 KiB pieces at odd destinations),
    so that body and output grow alike"""
    r = np.random.RandomState(seed)
    cases = dispatch_cases(seed)
    pick = {}
    for c in cases:
        if c[4] != "raw" and len(pick.setdefault(c[4], [])) < 12:
            pick[c[4]].append(c)
    b = BodyBuilder()
    for i, c in enumerate(x for v in pick.values() for x in v):
        b.add(c[0], c[1], c[2], c[3])
        if i % 5 == 0:
            n = 65536 + int(r.randint(1, 30000))
            b.add(255, n, _junk(r, n - int(r.randint(0, 3))))
    while b.len < (1 << 20):
        n = int(r.randint(1, 140000))
        b.add(255, n, _junk(r, n))
    b.add(UNKNOWN, 5, _junk(r, 333))
    return b.bytes(), b.out


@pytest.mark.gpu
def test_past_4gib(eng):
    """a ~1 MiB unit of packages from every class tiled past 2^32 + 1 MiB bytes of body and of output: device
    index, decode, block-wise comparison on the device with the unit's model output (peak ~9 GiB)"""
    import torch
    unit, unit_size = _big_unit(61)
    want, st, pkgs = model(unit, unit_size)
    reps = -(-((1 << 32) + (1 << 20)) // min(len(unit), unit_size)) + 1
    size = unit_size * reps
    torch.cuda.reset_peak_memory_stats()
    t_unit = torch.frombuffer(bytearray(unit), dtype=torch.uint8).cuda()
    t_body = t_unit.repeat(reps)
    assert t_body.numel() > (1 << 32) + (1 << 20) and size > (1 << 32) + (1 << 20)
    tab = _device_table(eng, t_body, size)
    n = len(tab)
    src_end = int((tab["src_off"] + tab["comp_len"]).max())
    dst_end = int((tab["dst_off"] + tab["out_len"]).max())
    assert src_end > (1 << 32) and dst_end > (1 << 32), (src_end, dst_end)
    assert set(entry_classes(tab[:n // reps])) == set(CLASS_TYPES)
    out = _prefilled(size)
    _, status = eng.decompress_device(t_body, size, out=out)
    assert status == [st[0] * reps, st[1] * reps]
    _tile_check(out, torch.frombuffer(bytearray(want), dtype=torch.uint8).cuda(), reps)
    assert (out[size:] == FILL).all()
    peak = torch.cuda.max_memory_allocated()
    print("past_4gib: body %d, output %d bytes, %d entries, peak %.2f GiB" % (t_body.numel(), size, n, peak / 2**30))
    del out, t_body, t_unit
    torch.cuda.empty_cache()
