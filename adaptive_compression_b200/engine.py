"""Functional layer over the C-ABI: torch is used only for device buffers and streams."""
import ctypes as C

import numpy as np
import torch

from . import _lib as L

FIXED_MARKER = b"\xff\xff\x00\x00"  # adaptive_compressor.py:303-310 (_find_marker is a stub)


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("adaptive_compression_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return L.lib()


def _stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def to_device(data):
    """bytes / bytearray / numpy uint8 -> 1-D uint8 cuda tensor"""
    if isinstance(data, torch.Tensor):
        return data.to("cuda", torch.uint8).contiguous().view(-1)
    a = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, np.uint8)
    if a.size == 0:
        return torch.empty(0, dtype=torch.uint8, device="cuda")
    return torch.from_numpy(a.copy() if not a.flags.writeable else a).to("cuda")


def method_mask(ids):
    m = 0
    for i in ids:
        if 0 < i < 32:
            m |= 1 << i
    return m


class CompressOutput:
    __slots__ = ("body", "body_len", "n_chunks", "first_raw", "n_packages", "types", "comp_lens", "payload_bytes",
                 "usage", "packages", "_keep")


def compress_device(t_in, chunk=4096, mask=L.NATIVE_MASK, flags=0, marker=FIXED_MARKER, out=None, work=None):
    """device tensor -> CompressOutput (body is a device tensor view of length body_len)"""
    lib = require_cuda()
    n = t_in.numel()
    bound = lib.ambc_compress_bound(n, chunk, len(marker))
    wbytes = lib.ambc_compress_workspace_bytes(n, chunk)
    if out is None or out.numel() < bound:
        out = torch.empty(bound, dtype=torch.uint8, device="cuda")
    if work is None or work.numel() < wbytes:
        work = torch.empty(max(wbytes, 1), dtype=torch.uint8, device="cuda")
    res = L.CompressResult()
    L.check(lib.ambc_compress_dev(C.c_void_p(t_in.data_ptr() if n else 0), n, chunk, mask, flags, marker, len(marker),
                                  C.c_void_p(out.data_ptr()), out.numel(), C.c_void_p(work.data_ptr()), work.numel(),
                                  C.byref(res), _stream_ptr()))
    o = CompressOutput()
    o.body = out[:res.body_len]
    o.body_len = res.body_len
    o.n_chunks = res.n_chunks
    o.first_raw = res.first_raw
    o.n_packages = res.n_packages
    o.payload_bytes = res.payload_bytes
    o.usage = list(res.usage)
    nc = res.n_chunks
    o.types = work[res.map_type_off:res.map_type_off + nc]
    o.comp_lens = work[res.map_comp_off:res.map_comp_off + 4 * nc].view(torch.int32)
    o._keep = (out, work)
    return o


def compress_dynamic_device(t_in, candidates, mask=L.NATIVE_MASK, flags=0, marker=FIXED_MARKER):
    """multi-candidate mode (adaptive_compressor.py:548-584): device tensor -> CompressOutput whose
    `packages` is the reference's package walk [(type, orig, comp)]"""
    lib = require_cuda()
    n = t_in.numel()
    cands = sorted({int(c) for c in candidates}, reverse=True)
    arr = (C.c_uint32 * len(cands))(*cands)
    wbytes = lib.ambc_compress_dynamic_workspace_bytes(n, arr, len(cands))
    if wbytes == 0:
        raise L.AmbcError(L.E_ARG, lib.ambc_last_error().decode("utf-8", "replace"))
    g = 0
    for c in cands:
        g = c if g == 0 else __import__("math").gcd(g, c)
    bound = n + (n // g + 3) * (len(marker) + 14) + len(marker) + 12 + 64
    out = torch.empty(bound, dtype=torch.uint8, device="cuda")
    work = torch.empty(max(wbytes, 1), dtype=torch.uint8, device="cuda")
    cap = n // g + 3
    info = (L.ChunkInfo * cap)()
    res = L.CompressResult()
    L.check(lib.ambc_compress_dynamic_dev(C.c_void_p(t_in.data_ptr() if n else 0), n, arr, len(cands), mask, flags, marker,
                                          len(marker), C.c_void_p(out.data_ptr()), out.numel(), C.c_void_p(work.data_ptr()),
                                          work.numel(), C.byref(res), info, cap, _stream_ptr()))
    o = CompressOutput()
    o.body = out[:res.body_len]
    o.body_len = res.body_len
    o.n_chunks = res.n_chunks
    o.first_raw = res.first_raw
    o.n_packages = res.n_packages
    o.payload_bytes = res.payload_bytes
    o.usage = list(res.usage)
    o.types = o.comp_lens = None
    o.packages = [(int(info[k].type), int(info[k].orig_len), int(info[k].comp_len)) for k in range(int(res.n_packages))]
    o._keep = (out, work)
    return o


# ---- one rank's input range of the multi-candidate mode (ambc_dyn_range_*) -------------------------------------
def _cands(candidates):
    cands = sorted({int(c) for c in candidates}, reverse=True)
    return cands, (C.c_uint32 * len(cands))(*cands)


class DynRange:
    """a rank's walked range (ambc_dyn_range_walk): the workspace, the buffer it was walked on and the entry table
    [(entry, status, exit, stop)] (exit / stop None when absent)"""
    __slots__ = ("r", "work", "buf", "table", "__weakref__")

    def __del__(self):
        if getattr(self, "r", None) is not None and L._lib is not None:
            L._lib.ambc_dyn_range_free(C.byref(self.r))


def _dyn_row(e):
    none = lambda v: None if v == L.DYN_NONE else int(v)  # noqa: E731
    return (int(e.entry), int(e.status), none(e.exit), none(e.stop))


def dyn_range_walk(t_buf, lo, hi, n, candidates, mask=L.NATIVE_MASK, flags=0, marker_bytes=4, work=None):
    """phase 1 on input [lo, hi): t_buf = input[lo, min(n, hi + 8192)) as a device tensor -> DynRange"""
    lib = require_cuda()
    _, arr = _cands(candidates)
    wbytes = lib.ambc_dyn_range_workspace_bytes(lo, hi, n, arr, len(arr))
    if wbytes == 0:
        raise L.AmbcError(L.E_ARG, lib.ambc_last_error().decode("utf-8", "replace"))
    if work is None or work.numel() < wbytes:
        work = torch.empty(int(wbytes), dtype=torch.uint8, device="cuda")
    dr = DynRange()
    dr.r = L.DynRange()
    tab = (L.DynEntry * L.DYN_MAX_ENTRIES)()
    nt = C.c_uint32(0)
    rc = lib.ambc_dyn_range_walk(C.c_void_p(t_buf.data_ptr() if t_buf.numel() else 0), t_buf.numel(), lo, hi, n, arr,
                                 len(arr), mask, flags, marker_bytes, C.c_void_p(work.data_ptr()), work.numel(),
                                 C.byref(dr.r), tab, L.DYN_MAX_ENTRIES, C.byref(nt), _stream_ptr())
    L.check(rc)
    dr.work, dr.buf = work, t_buf
    dr.table = [_dyn_row(tab[k]) for k in range(nt.value)]
    return dr


def dyn_range_resolve(dr, entry):
    """phase 2: stitch the chain from an unresolved entry until it leaves the range or stops -> its updated row
    (also stored in dr.table)"""
    out = L.DynEntry()
    L.check(require_cuda().ambc_dyn_range_resolve(C.byref(dr.r), entry, C.byref(out), _stream_ptr()))
    row = _dyn_row(out)
    dr.table = [row if t[0] == entry else t for t in dr.table]
    return row


def dyn_range_encode(dr, entry, marker=FIXED_MARKER, out=None):
    """phase 3: the rank's packages of the chain from its true entry -> (fragment device tensor, stop or None,
    [(pos, type, orig, comp)] with global positions, usage [raw, 1..4], payload bytes)"""
    lib = require_cuda()
    r = dr.r
    n_pos = max((r.hi - r.lo) // 256 + 2, 1)
    bound = (r.hi - r.lo) + 8192 + n_pos * (len(marker) + 14) + 64
    if out is None or out.numel() < bound:
        out = torch.empty(bound, dtype=torch.uint8, device="cuda")
    info = (L.ChunkInfo * n_pos)()
    res = L.CompressResult()
    stop = C.c_uint64(0)
    L.check(lib.ambc_dyn_range_encode(C.byref(r), C.c_void_p(dr.buf.data_ptr() if dr.buf.numel() else 0), entry, marker,
                                      len(marker), C.c_void_p(out.data_ptr()), out.numel(), C.byref(res), info, n_pos,
                                      C.byref(stop), _stream_ptr()))
    pk = [(int(info[k].pos), int(info[k].type), int(info[k].orig_len), int(info[k].comp_len))
          for k in range(int(res.n_packages))]
    return (out[:res.body_len], None if stop.value == L.DYN_NONE else int(stop.value), pk, list(res.usage),
            int(res.payload_bytes))


def package_map(o, n, chunk, per_chunk_raw=False):
    """[(type, orig, comp)] per package, as the reference's package walk would list them"""
    types = o.types.cpu().numpy()
    comps = o.comp_lens.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    pm = []
    for i in range(int(o.n_chunks)):
        orig = min(chunk, n - i * chunk)
        if not per_chunk_raw and o.first_raw >= 0 and i >= o.first_raw:
            rest = n - i * chunk
            pm.append((255, rest, rest))
            break
        t = int(types[i])
        pm.append((t, orig, int(comps[i]) if t != 255 else orig))
    return pm


def index_host(body, orig_size, marker=FIXED_MARKER, known_mask=L.NATIVE_MASK):
    """host package walk -> (numpy structured table, covered bytes)"""
    lib = L.lib()
    b = np.frombuffer(body, dtype=np.uint8) if not isinstance(body, np.ndarray) else body
    ne, cov = C.c_uint64(0), C.c_uint64(0)
    ptr = C.c_void_p(b.ctypes.data if b.size else 0)
    L.check(lib.ambc_index_host(ptr, b.size, marker, len(marker), orig_size, known_mask, None, 0,
                                C.byref(ne), C.byref(cov)))
    table = np.zeros(max(ne.value, 1), dtype=np.dtype([("src_off", "<u8"), ("dst_off", "<u8"), ("comp_len", "<u4"),
                                                        ("orig_len", "<u4"), ("type", "<u4"), ("out_len", "<u4")]))
    L.check(lib.ambc_index_host(ptr, b.size, marker, len(marker), orig_size, known_mask,
                                C.c_void_p(table.ctypes.data), ne.value, C.byref(ne), C.byref(cov)))
    return table[:ne.value], cov.value


def index_device(t_body, orig_size, marker=FIXED_MARKER, known_mask=L.NATIVE_MASK):
    """package table built on the GPU -> (uint8 device tensor of 32-byte entries, n entries, covered bytes)"""
    lib = require_cuda()
    ne, cov = C.c_uint64(0), C.c_uint64(0)
    ptr = C.c_void_p(t_body.data_ptr() if t_body.numel() else 0)
    L.check(lib.ambc_index_dev(ptr, t_body.numel(), marker, len(marker), orig_size, known_mask, None, 0,
                               C.byref(ne), C.byref(cov), _stream_ptr()))
    t_table = torch.empty(max(ne.value, 1) * 32, dtype=torch.uint8, device="cuda")
    if ne.value:
        L.check(lib.ambc_index_dev(ptr, t_body.numel(), marker, len(marker), orig_size, known_mask,
                                   C.c_void_p(t_table.data_ptr()), ne.value, C.byref(ne), C.byref(cov), _stream_ptr()))
    return t_table, ne.value, cov.value


def decompress_device(t_body, orig_size, marker=FIXED_MARKER, known_mask=L.NATIVE_MASK, body_host=None, out=None,
                      gpu_index=None):
    """device body -> (device output tensor, status [codec errors, length mismatches]).
    The package table comes from the GPU index (default when no host copy of the body is given)
    or from the host walk."""
    lib = require_cuda()
    if gpu_index is None:
        gpu_index = body_host is None
    if out is None or out.numel() < orig_size:
        out = torch.empty(max(orig_size, 1), dtype=torch.uint8, device="cuda")
    status = torch.zeros(2, dtype=torch.int32, device="cuda")
    if gpu_index:
        t_table, n_table, _ = index_device(t_body, orig_size, marker, known_mask)
        table = range(n_table)
    else:
        if body_host is None:
            body_host = t_body.cpu().numpy()
        table, _ = index_host(body_host, orig_size, marker, known_mask)
        t_table = torch.from_numpy(table.view(np.uint8).reshape(-1).copy()).to("cuda") if len(table) else \
            torch.empty(0, dtype=torch.uint8, device="cuda")
    L.check(lib.ambc_decompress_dev_mask(C.c_void_p(t_body.data_ptr() if t_body.numel() else 0), t_body.numel(),
                                         C.c_void_p(t_table.data_ptr() if len(table) else 0), len(table),
                                         C.c_void_p(out.data_ptr()), orig_size, known_mask, C.c_void_p(status.data_ptr()),
                                         _stream_ptr()))
    torch.cuda.current_stream().synchronize()
    return out[:orig_size], status.cpu().tolist()


# ---- range-local index (ambc_range_*): one byte range [lo, hi) of a body per rank -------------------------
class RangeIndex:
    """the phase-1 tables of one range (ambc_range_index) and the workspace that holds them"""
    __slots__ = ("r", "work", "marker")


def range_index(t_buf, lo, hi, body_len, orig_size, marker=FIXED_MARKER, known_mask=L.NATIVE_MASK, work=None):
    """phase 1 on body[lo, hi): t_buf = body[lo, min(hi + len(marker) + 13, body_len)) (the range and the header
    halo, distributed.buffer_span) as a device tensor -> RangeIndex"""
    lib = require_cuda()
    r = L.Range()
    guess = int(lib.ambc_range_workspace_bytes(hi - lo, (hi - lo) // 2048 + 64))
    if work is None or work.numel() < guess:
        work = torch.empty(guess, dtype=torch.uint8, device="cuda")
    while True:
        rc = lib.ambc_range_index(C.c_void_p(t_buf.data_ptr() if t_buf.numel() else 0), t_buf.numel(), lo, hi, body_len,
                                  marker, len(marker), orig_size, known_mask, C.c_void_p(work.data_ptr()), work.numel(),
                                  C.byref(r), _stream_ptr())
        if rc == L.E_CAPACITY and r.work_bytes > work.numel():
            work = torch.empty(int(r.work_bytes), dtype=torch.uint8, device="cuda")
            continue
        L.check(rc)
        break
    ri = RangeIndex()
    ri.r, ri.work, ri.marker = r, work, marker
    return ri


def range_init_state():
    """the walk's state before body position 0"""
    return L.RangeState(0, 0, L.RANGE_NO_PKG, 0, 0, 0, 0, L.RANGE_RUNNING)


def range_fold(ri, state):
    """phase 2, one step: the walk's state behind this range given the state before it"""
    out = L.RangeState()
    L.check(require_cuda().ambc_range_fold(C.byref(ri.r), C.byref(state), C.byref(out), _stream_ptr()))
    return out


def range_table(ri, entry, count_only=False):
    """phase 3: -> (uint8 device tensor of 32-byte ambc_pkg entries, n entries, out_lo, out_hi, need).
    src_off is relative to the range's buffer, dst_off to out_lo; `need` = payload bytes past the halo
    that the buffer must hold before decoding"""
    lib = require_cuda()
    ne, olo, ohi, need = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    L.check(lib.ambc_range_table(C.byref(ri.r), C.byref(entry), None, 0, C.byref(ne), C.byref(olo), C.byref(ohi),
                                 C.byref(need), _stream_ptr()))
    t_table = torch.empty(max(ne.value, 1) * 32, dtype=torch.uint8, device="cuda")
    if ne.value and not count_only:
        L.check(lib.ambc_range_table(C.byref(ri.r), C.byref(entry), C.c_void_p(t_table.data_ptr()), ne.value, C.byref(ne),
                                     C.byref(olo), C.byref(ohi), C.byref(need), _stream_ptr()))
    return t_table, ne.value, olo.value, ohi.value, need.value


def range_out_offset(state, lo, orig_size, marker_bytes=4, known_mask=L.NATIVE_MASK):
    """first output byte owned by the range starting at body position lo, given the state the fold handed to it
    (host arithmetic, no device needed)"""
    return int(L.lib().ambc_range_out_offset(C.byref(state), lo, orig_size, marker_bytes, known_mask))


def range_decode(t_buf, t_table, n_entries, out_len, known_mask=L.NATIVE_MASK, out=None):
    """decode a range's table into its output slice of out_len bytes -> (slice, status [codec errors, length
    mismatches]); the zero tail is written when the slice reaches past the last entry"""
    lib = require_cuda()
    if out is None or out.numel() < out_len:
        out = torch.empty(max(out_len, 1), dtype=torch.uint8, device="cuda")
    status = torch.zeros(2, dtype=torch.int32, device="cuda")
    L.check(lib.ambc_decompress_dev_mask(C.c_void_p(t_buf.data_ptr() if t_buf.numel() else 0), t_buf.numel(),
                                         C.c_void_p(t_table.data_ptr() if n_entries else 0), n_entries,
                                         C.c_void_p(out.data_ptr()), out_len, known_mask, C.c_void_p(status.data_ptr()),
                                         _stream_ptr()))
    torch.cuda.current_stream().synchronize()
    return out[:out_len], status.cpu().tolist()


def _pack_items(items):
    offs = np.zeros(len(items) + 1, dtype=np.uint64)
    for i, it in enumerate(items):
        offs[i + 1] = offs[i] + len(it)
    blob = np.frombuffer(b"".join(bytes(x) for x in items), dtype=np.uint8)
    return blob, offs


def codec_encode_batch(method, items):
    """items: list of bytes (each <= 8192).  -> list of bytes | int error code"""
    lib = require_cuda()
    if not items:
        return []
    if max(len(x) for x in items) > L.MAX_CODEC_CHUNK:
        raise L.AmbcError(L.E_TOO_LARGE, "codec items are limited to %d bytes" % L.MAX_CODEC_CHUNK)
    blob, offs = _pack_items(items)
    stride = int(lib.ambc_codec_bound(method, max(len(x) for x in items) or 1))
    stride = (stride + 15) & ~15
    t_in = to_device(blob)
    t_off = torch.from_numpy(offs.view(np.int64)).to("cuda")
    t_out = torch.empty(stride * len(items), dtype=torch.uint8, device="cuda")
    t_len = torch.empty(len(items), dtype=torch.int32, device="cuda")
    L.check(lib.ambc_codec_encode_batch(method, C.c_void_p(t_in.data_ptr() if blob.size else 0),
                                        C.c_void_p(t_off.data_ptr()), len(items), C.c_void_p(t_out.data_ptr()),
                                        stride, C.c_void_p(t_len.data_ptr()), _stream_ptr()))
    lens = t_len.cpu().numpy()
    outs = t_out.cpu().numpy()
    return [int(l) if l < 0 else outs[i * stride:i * stride + int(l)].tobytes() for i, l in enumerate(lens)]


def codec_decode_batch(method, items, orig_lens):
    """items: payloads; -> list of bytes | int error code (what the reference's decompress returns)"""
    require_cuda()
    if not items:
        return []
    stride = (max(max(orig_lens), 1) + 512 + 15) & ~15
    if method == L.DEFLATE:
        stride += 32768  # window of a stream that runs past original_length (it is checked to its end, then truncated)
    elif method == L.LZMA:
        stride += 65536  # the whole stride is the dictionary: a stream is decoded (and its check verified) to its end
    out = _codec_decode(method, items, orig_lens, stride)
    # LZMA streams that decode past the stride: again, one at a time, with room for them
    for i, o in enumerate(out):
        room = stride
        while o == L.E_CAPACITY:
            room *= 4
            if room > (1 << 34):
                raise L.AmbcError(L.E_CAPACITY, "stream %d decodes to more than %d bytes" % (i, 1 << 34))
            o = _codec_decode(method, [items[i]], [orig_lens[i]], room)[0]
        out[i] = o
    return out


def _codec_decode(method, items, orig_lens, stride):
    lib = L.lib()
    blob, offs = _pack_items(items)
    t_in = to_device(blob)
    t_off = torch.from_numpy(offs.view(np.int64)).to("cuda")
    t_orig = torch.tensor(list(orig_lens), dtype=torch.int32, device="cuda")
    t_out = torch.zeros(stride * len(items), dtype=torch.uint8, device="cuda")
    t_len = torch.empty(len(items), dtype=torch.int32, device="cuda")
    L.check(lib.ambc_codec_decode_batch(method, C.c_void_p(t_in.data_ptr() if blob.size else 0),
                                        C.c_void_p(t_off.data_ptr()), C.c_void_p(t_orig.data_ptr()), len(items),
                                        C.c_void_p(t_out.data_ptr()), stride, C.c_void_p(t_len.data_ptr()),
                                        _stream_ptr()))
    lens = t_len.cpu().numpy()
    outs = t_out.cpu().numpy()
    return [int(l) if l < 0 else outs[i * stride:i * stride + int(l)].tobytes() for i, l in enumerate(lens)]


def should_use_batch(items):
    """-> (list of {method id: bool}, list of entropies)"""
    lib = require_cuda()
    if not items:
        return [], []
    if max(len(x) for x in items) > L.MAX_CODEC_CHUNK:
        raise L.AmbcError(L.E_TOO_LARGE, "codec items are limited to %d bytes" % L.MAX_CODEC_CHUNK)
    blob, offs = _pack_items(items)
    t_in = to_device(blob)
    t_off = torch.from_numpy(offs.view(np.int64)).to("cuda")
    t_g = torch.zeros(len(items), dtype=torch.uint8, device="cuda")
    t_h = torch.zeros(len(items), dtype=torch.float64, device="cuda")
    L.check(lib.ambc_should_use_batch(C.c_void_p(t_in.data_ptr() if blob.size else 0), C.c_void_p(t_off.data_ptr()),
                                      len(items), C.c_void_p(t_g.data_ptr()), C.c_void_p(t_h.data_ptr()),
                                      _stream_ptr()))
    g = t_g.cpu().numpy()
    return [{m: bool((int(x) >> m) & 1) for m in (1, 2, 3, 4)} for x in g], t_h.cpu().tolist()


def find_marker_device(t_in, max_len=32):
    """-> (marker bytes left-aligned, length in bits); raises ValueError when none (marker_finder.py:123)"""
    lib = require_cuda()
    ln, val = C.c_uint32(0), C.c_uint64(0)
    L.check(lib.ambc_find_marker_dev(C.c_void_p(t_in.data_ptr() if t_in.numel() else 0), t_in.numel(), max_len,
                                     C.byref(ln), C.byref(val), _stream_ptr()))
    return marker_bytes(val.value, ln.value), ln.value


def marker_bytes(value, length):
    """left-aligned, zero padded to a byte boundary (marker_finder.py:100-110)"""
    nb = (length + 7) // 8
    return (value << (8 * nb - length)).to_bytes(nb, "big")


def synth(n, offset=0, seed=0xA3BC0001, kind_mask=0b1011111, out=None):
    """n bytes of the synthetic corpus starting at byte `offset` -> device tensor"""
    lib = require_cuda()
    if out is None:
        out = torch.empty(n, dtype=torch.uint8, device="cuda")
    L.check(lib.ambc_synth_dev(C.c_void_p(out.data_ptr() if n else 0), offset, n, seed, kind_mask, _stream_ptr()))
    return out[:n]


# ---- pinned host buffers for the file API (grow-only cache: pinning a GiB costs a few 100 ms) ----------
_PINNED = {}


def pinned(slot, nbytes):
    """numpy uint8 view of at least `nbytes` bytes of page-locked host memory (one buffer per slot name)"""
    lib = require_cuda()
    cur = _PINNED.get(slot)
    if cur is None or cur[1] < nbytes:
        if cur is not None:
            lib.ambc_host_free(C.c_void_p(cur[0]))
            _PINNED.pop(slot)
        cap = max(int(nbytes), 1 << 20)
        cap += cap >> 3
        ptr = lib.ambc_host_alloc(cap)
        if not ptr:
            raise L.AmbcError(L.E_CUDA, lib.ambc_last_error().decode("utf-8", "replace"))
        _PINNED[slot] = cur = (int(ptr), cap)
    return np.ctypeslib.as_array((C.c_uint8 * cur[1]).from_address(cur[0]))


def compress_host(h_in, n, chunk, mask=L.NATIVE_MASK, flags=0, marker=FIXED_MARKER):
    """host buffer -> (body view in the pinned 'body' slot, CompressResult, types u8[], comp_lens u32[]) through
    ambc_compress_host (piece-wise upload overlapping the chunk kernels, body downloaded piece by piece)"""
    lib = require_cuda()
    bound = int(lib.ambc_compress_bound(n, chunk, len(marker)))
    n_chunks = (n + chunk - 1) // chunk
    body = pinned("body", bound)
    types = np.empty(max(n_chunks, 1), dtype=np.uint8)
    comps = np.empty(max(n_chunks, 1), dtype=np.uint32)
    res = L.CompressResult()
    L.check(lib.ambc_compress_host(C.c_void_p(h_in.ctypes.data if n else 0), n, chunk, mask, flags, marker, len(marker),
                                   C.c_void_p(body.ctypes.data), bound, C.c_void_p(types.ctypes.data),
                                   C.c_void_p(comps.ctypes.data), C.byref(res)))
    return body[:res.body_len], res, types[:n_chunks], comps[:n_chunks]


def decompress_host(h_body, orig_size, marker=FIXED_MARKER, known_mask=L.NATIVE_MASK):
    """host body -> (output view in the pinned 'out' slot, status) through ambc_decompress_host"""
    lib = require_cuda()
    out = pinned("out", max(int(orig_size), 1))
    st = (C.c_uint32 * 2)()
    L.check(lib.ambc_decompress_host(C.c_void_p(h_body.ctypes.data if h_body.size else 0), int(h_body.size), marker,
                                     len(marker), known_mask, C.c_void_p(out.ctypes.data), int(orig_size), st))
    return out[:orig_size], [int(st[0]), int(st[1])]
