"""GPU parity of the chunk trial at its decision boundaries: the cases of tests/trial_edges.py (built and checked on
the CPU by test_cpu_trial_edges.py) run through every kernel that runs sf_select -- k_select_fast<4096 | 8192> on
the fixed grid (per-chunk-raw and strict), k_dynamic_walk + k_select_span_fast in the multi-candidate mode, and the
plug-in batch kernels (should_use, encode) -- and are compared with the oracle.  Output and work buffers are filled
with a poison byte before every call, and every GPU body is decoded back to its input."""
import ctypes as C
import math

import numpy as np
import pytest

import oracle as O
import trial_edges as T

pytestmark = pytest.mark.gpu

POISON = 0xA5


@pytest.fixture(scope="module")
def eng():
    from adaptive_compression_b200 import engine
    engine.require_cuda()
    return engine


def _full(n):
    import torch
    return torch.full((max(int(n), 1),), POISON, dtype=torch.uint8, device="cuda")


def groups():
    """(chunk, methods, marker) -> [Case] of the single-chunk cases"""
    g = {}
    for c, _ in T.cases():
        if isinstance(c.chunk, int):
            g.setdefault((c.chunk, tuple(c.methods), c.marker), []).append(c)
    return g


def files(cases, chunk):
    """the group's full chunks in one file, and every short chunk as the last chunk of a file behind the first full one"""
    full = [c.data for c in cases if len(c.data) == chunk]
    out = [b"".join(full)] if full else []
    lead = full[0] if full else b""
    out += [lead + c.data for c in cases if len(c.data) < chunk]
    return out


def fixed(eng, data, chunk, methods, marker, pcr):
    from adaptive_compression_b200 import _lib as L
    lib = L.lib()
    n = len(data)
    t = eng.to_device(data)
    out = _full(lib.ambc_compress_bound(n, chunk, len(marker)))
    work = _full(lib.ambc_compress_workspace_bytes(n, chunk))
    return eng.compress_device(t, chunk, eng.method_mask(methods), L.F_PER_CHUNK_RAW if pcr else 0, marker, out=out,
                               work=work)


def usage_of(pm):
    u = [0] * 5
    for t, _, _ in pm:
        u[t if 1 <= t <= 4 else 0] += 1
    return u


def check_fixed(eng, data, chunk, methods, marker, pcr, bad, tag):
    o = fixed(eng, data, chunk, methods, marker, pcr)
    body = o.body.cpu().numpy().tobytes()
    wbody, wpm = O.compress_body(data, chunk, methods, marker, per_chunk_raw=pcr)
    pm = [tuple(p) for p in eng.package_map(o, len(data), chunk, pcr)]
    wpm = [tuple(p) for p in wpm]
    if pm != wpm:
        bad.append((tag, "packages", [(i, a, b) for i, (a, b) in enumerate(zip(pm, wpm)) if a != b][:4], len(pm), len(wpm)))
        return None
    if body != wbody:
        bad.append((tag, "body", next(i for i, (a, b) in enumerate(zip(body + b"\0", wbody + b"\1")) if a != b)))
        return None
    if o.n_packages != len(wpm) or o.usage != usage_of(wpm) or o.payload_bytes != sum(p[2] for p in wpm if p[0] != 255):
        bad.append((tag, "counters", o.n_packages, o.usage, o.payload_bytes, len(wpm), usage_of(wpm)))
    if not pcr:
        first = next((i for i, p in enumerate(wpm) if p[0] == 255), -1)
        if o.first_raw != first:
            bad.append((tag, "first_raw", o.first_raw, first))
    dec, status = eng.decompress_device(o.body, len(data), marker=marker)
    if status != [0, 0] or dec.cpu().numpy().tobytes() != data:
        bad.append((tag, "decode", status))
    return o


def test_fixed_grid_per_chunk_raw(eng):
    """every group's chunks in one file: types, lengths, body, counters equal the oracle's, body decodes"""
    bad, seen = [], set()
    for (chunk, methods, marker), cases in groups().items():
        for k, data in enumerate(files(cases, chunk)):
            check_fixed(eng, data, chunk, methods, marker, True, bad, (chunk, methods, len(marker), k))
        seen.add(T.inst(chunk))
    assert seen == {4096, 8192}
    assert not bad, bad[:10]


def test_fixed_grid_strict(eng):
    """strict mode: a losing boundary chunk first, in the middle and last, behind and in front of winners"""
    bad, placed = [], 0
    for (chunk, methods, marker), cases in groups().items():
        full = [c for c in cases if len(c.data) == chunk]
        outcome = {id(c): m["chosen"][0] for c, m in T.cases() if c in full}
        win = [c.data for c in full if outcome[id(c)] != 255]
        lose = [c.data for c in full if outcome[id(c)] == 255]
        for data in files(cases, chunk):
            check_fixed(eng, data, chunk, methods, marker, False, bad, (chunk, methods, len(marker), "group"))
        if not win or not lose:
            continue
        for L in lose:
            mid = len(win) // 2
            for data in (L + b"".join(win), b"".join(win[:mid]) + L + b"".join(win[mid:]), b"".join(win) + L):
                check_fixed(eng, data, chunk, methods, marker, False, bad, (chunk, methods, len(marker), "placed"))
                placed += 1
    assert placed > 0
    assert not bad, bad[:10]


def dynamic(eng, data, cands, methods, marker, pcr):
    """compress_dynamic_device with poisoned output and work buffers"""
    from adaptive_compression_b200 import _lib as L
    lib = eng.require_cuda()
    n = len(data)
    t = eng.to_device(data)
    cands = sorted({int(c) for c in cands}, reverse=True)
    arr = (C.c_uint32 * len(cands))(*cands)
    g = 0
    for c in cands:
        g = math.gcd(g, c)
    work = _full(lib.ambc_compress_dynamic_workspace_bytes(n, arr, len(cands)))
    out = _full(n + (n // g + 3) * (len(marker) + 14) + len(marker) + 12 + 64)
    cap = n // g + 3
    info = (L.ChunkInfo * cap)()
    res = L.CompressResult()
    L.check(lib.ambc_compress_dynamic_dev(C.c_void_p(t.data_ptr()), n, arr, len(cands), eng.method_mask(methods),
                                          L.F_PER_CHUNK_RAW if pcr else 0, marker, len(marker), C.c_void_p(out.data_ptr()),
                                          out.numel(), C.c_void_p(work.data_ptr()), work.numel(), C.byref(res), info, cap,
                                          eng._stream_ptr()))
    pk = [(int(info[k].type), int(info[k].orig_len), int(info[k].comp_len)) for k in range(int(res.n_packages))]
    return out[:res.body_len], pk


def check_dynamic(eng, data, cands, methods, marker, pcr, bad, tag):
    body_t, pk = dynamic(eng, data, cands, methods, marker, pcr)
    wbody, wpm = O.compress_body(data, tuple(cands), methods, marker, per_chunk_raw=pcr)
    if pk != [tuple(p) for p in wpm]:
        bad.append((tag, "packages", pk[:4], wpm[:4]))
        return
    if body_t.cpu().numpy().tobytes() != wbody:
        bad.append((tag, "body"))
        return
    dec, status = eng.decompress_device(body_t, len(data), marker=marker)
    if status != [0, 0] or dec.cpu().numpy().tobytes() != data:
        bad.append((tag, "decode", status))


def test_multi_candidate_ratio_ties(eng):
    """equal (len + ovh) / size for two candidates: the larger keeps the tie; one RLE run either side flips it"""
    bad = []
    cases = [c for c, _ in T.cases() if c.label == "ratio_tie"]
    for c in cases:
        check_dynamic(eng, c.data, c.chunk, c.methods, c.marker, False, bad, (c.chunk, c.side))
    assert len(cases) == 6 and not bad, bad


def test_multi_candidate_single_sizes(eng):
    """the single-chunk cases of chunks <= 4096 under a one-size candidate list: k_dynamic_walk (SfCtx<8192>) chooses,
    k_select_span_fast<4096> encodes"""
    bad, n = [], 0
    for (chunk, methods, marker), cases in groups().items():
        if chunk > 4096 or chunk % 16 or chunk < 256:  # (sizes the multi-candidate mode takes)
            continue
        for data in files(cases, chunk):
            for pcr in (True, False):
                check_dynamic(eng, data, (chunk,), methods, marker, pcr, bad, (chunk, methods, len(marker), pcr))
                n += 1
    assert n and not bad, bad[:10]


def _datas():
    out, seen = [], set()
    for c, _ in T.cases():
        if 0 < len(c.data) <= 8192 and c.data not in seen:
            seen.add(c.data)
            out.append(c.data)
    return out


def test_should_use_batch(eng):
    """the gates of every case (RLE steps 1..8, n 4097..8192 included) and the exact entropy"""
    datas = _datas()
    gates, ent = eng.should_use_batch(datas)
    bad = []
    for d, g, h in zip(datas, gates, ent):
        want = [O.should_use(m, d) for m in (1, 2, 3, 4)]
        if [g[m] for m in (1, 2, 3, 4)] != want:
            bad.append((len(d), [g[m] for m in (1, 2, 3, 4)], want, h))
        if len(d) >= 100 and abs(h - O.entropy(d)) > 1e-12:
            bad.append((len(d), "entropy", h, O.entropy(d)))
    assert any(len(d) > 4096 for d in datas)
    assert not bad, bad[:10]


def encode_batch(eng, method, items):
    """engine.codec_encode_batch with a poisoned output buffer"""
    import torch
    from adaptive_compression_b200 import _lib as L
    lib = eng.require_cuda()
    blob, offs = eng._pack_items(items)
    stride = (int(lib.ambc_codec_bound(method, max(len(x) for x in items))) + 15) & ~15
    t_in = eng.to_device(blob)
    t_off = torch.from_numpy(offs.view(np.int64)).to("cuda")
    t_out = _full(stride * len(items))
    t_len = torch.full((len(items),), -12345, dtype=torch.int32, device="cuda")
    L.check(lib.ambc_codec_encode_batch(method, C.c_void_p(t_in.data_ptr()), C.c_void_p(t_off.data_ptr()), len(items),
                                        C.c_void_p(t_out.data_ptr()), stride, C.c_void_p(t_len.data_ptr()),
                                        eng._stream_ptr()))
    lens, outs = t_len.cpu().numpy(), t_out.cpu().numpy()
    return [int(v) if v < 0 else outs[i * stride:i * stride + int(v)].tobytes() for i, v in enumerate(lens)]


@pytest.mark.parametrize("mid", [1, 2, 3])
def test_codec_encode_batch(eng, mid):
    datas = _datas()
    got = encode_batch(eng, mid, datas)
    bad = [(i, len(d)) for i, (d, g) in enumerate(zip(datas, got)) if g != O.compress(mid, d, lz_fast=True)]
    assert not bad, bad[:10]
