"""File -> file compress and decompress through fixed-size device windows (DESIGN.md §4.6).

The in-memory paths of AdaptiveCompressor hold the whole file on one GPU.  Here the file is cut into windows that
are processed one after another with the range calls the multi-GPU paths use across ranks (distributed.py): the
fold that joins ranks carries the state from window k to window k + 1, so device memory and pinned host memory are
bounded by the window size W, not by the file size, and the bytes written are those of the in-memory path.

  compress_fixed    windows of whole chunks through ambc_compress_dev; the END package of every window but the last
                    is dropped, the first chunk without a winner turns the rest of the file into one raw package.
  compress_dynamic  windows of whole 64 * g segments through ambc_dyn_range_walk / _resolve / _encode; the exit of
                    window k is the entry of window k + 1.
  decompress        body windows through ambc_range_index / _fold / _table; each window's table is decoded in pieces
                    whose output fits a budget.
  find_marker       MarkerFinder.find_marker over the windows: one pass per level, the flags accumulated with the
                    carry bits of the bytes before each window.

Reading (and hashing) window k + 1 and its upload on a side stream, the kernels of window k and the download and
write of window k - 1 overlap: a reader, a hasher and an uploader thread feed the main thread, a writer (and, for
decompress, a hasher) drain it.  Every thread is joined before a driver returns, on errors too."""
import ctypes as C
import hashlib
import os
import queue
import threading

import numpy as np
import torch

from . import _lib as L
from . import distributed as D
from . import engine

RING = 3                 # pinned host slots per direction
DEV_SLOTS = 2            # device input slots: window k + 1 uploads while window k computes
STAGE = 64 << 20         # pinned staging for payload bytes a decoded package needs behind a window's halo
_POLL = 0.05
_ZEROS = np.zeros(1 << 20, dtype=np.uint8)


class _Stop(Exception):
    """raised in a thread blocked on a queue once the flow is aborted"""


class _Flow:
    """threads of one driver call: the first error aborts all of them; close() joins every thread"""

    def __init__(self):
        self.abort = threading.Event()
        self.errors = []
        self.threads = []
        self.closers = []

    def get(self, q):
        while True:
            try:
                return q.get(timeout=_POLL)
            except queue.Empty:
                if self.abort.is_set():
                    raise _Stop()

    def spawn(self, fn):
        def run():
            try:
                fn()
            except _Stop:
                pass
            except BaseException as e:  # noqa: B902 -- handed to the main thread by check()
                self.errors.append(e)
                self.abort.set()
        th = threading.Thread(target=run, daemon=True)
        th.start()
        self.threads.append(th)

    def check(self):
        if self.errors:
            raise self.errors[0]

    def join(self, threads=None):
        """wait for the threads (all by default) to finish their work, the normal end; then report a thread's error"""
        for th in (self.threads if threads is None else threads):
            while th.is_alive():
                th.join(_POLL)
                if self.errors:
                    break
        self.check()

    def on_close(self, fn):
        """fn() runs in close(), once every thread has ended (a file descriptor the threads read from, say)"""
        self.closers.append(fn)

    def close(self):
        self.abort.set()
        for th in self.threads:
            th.join()
        for fn in self.closers:
            fn()


class _Slot:
    """one pinned host buffer, back on its free list once every consumer has released it"""

    def __init__(self, free, nbytes):
        self.free = free
        self.t = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, pin_memory=True)
        self.lock = threading.Lock()
        self.pending = 0

    def ensure(self, nbytes):
        if self.t.numel() < nbytes:
            self.t = torch.empty(int(nbytes), dtype=torch.uint8, pin_memory=True)
        return self

    def hold(self, k):
        with self.lock:
            self.pending += k

    def release(self):
        with self.lock:
            self.pending -= 1
            done = self.pending == 0
        if done:
            self.free.put(self)


def _ring(n, nbytes):
    free = queue.Queue()
    for _ in range(n):
        free.put(_Slot(free, nbytes))
    return free


def _pread(fd, view, off):
    pos = 0
    while pos < len(view):
        got = os.preadv(fd, [view[pos:]], off + pos)
        if not got:
            raise IOError("short read at offset %d" % (off + pos))
        pos += got


class _Source:
    """reads spans (offset, length, hash_len) of a file in order into a ring of pinned slots; the first hash_len
    bytes of every span go through MD5 in file order; each span is uploaded into one of DEV_SLOTS device buffers on
    a side stream.  The main thread takes (index, device view, tail) from next(): tail = the span's last <= 4 bytes.
    After passthrough() the spans are no longer uploaded: next() hands out the pinned slot instead (release it)."""

    def __init__(self, flow, path, spans, slot_bytes, hash_input=False):
        self.flow, self.spans = flow, spans
        self.md5 = hashlib.md5() if hash_input else None
        self.host_free = _ring(RING, slot_bytes)
        self.dev_free = queue.Queue()
        for _ in range(DEV_SLOTS):
            self.dev_free.put(torch.empty(max(int(slot_bytes), 1), dtype=torch.uint8, device="cuda"))
        self.q_hash, self.q_up, self.q_ready = queue.Queue(), queue.Queue(), queue.Queue()
        self.copy_stream = torch.cuda.Stream()
        self.device = torch.cuda.current_device()
        self._through = threading.Event()
        self.fd = fd = os.open(path, os.O_RDONLY)
        flow.on_close(lambda: os.close(fd))  # (not self: a cycle would keep the device slots until a GC pass)
        flow.spawn(self._read)
        if self.md5 is not None:
            flow.spawn(self._hash)
        flow.spawn(self._upload)

    def _read(self):
        for k, (off, ln, hl) in enumerate(self.spans):
            slot = self.flow.get(self.host_free).ensure(ln)
            slot.hold(2 if self.md5 is not None else 1)
            view = memoryview(slot.t.numpy())[:ln]
            _pread(self.fd, view, off)
            tail = bytes(view[max(0, ln - 4):ln])
            if self.md5 is not None:
                self.q_hash.put((slot, ln, hl))
            self.q_up.put((k, slot, ln, tail))

    def _hash(self):
        for _ in self.spans:
            slot, ln, hl = self.flow.get(self.q_hash)
            self.md5.update(memoryview(slot.t.numpy())[:hl])
            slot.release()

    def _upload(self):
        torch.cuda.set_device(self.device)
        for _ in self.spans:
            k, slot, ln, tail = self.flow.get(self.q_up)
            if self._through.is_set():
                self.q_ready.put((k, None, slot, ln, tail))
                continue
            dev = self.flow.get(self.dev_free)
            if dev.numel() < ln:
                dev = torch.empty(ln, dtype=torch.uint8, device="cuda")
            with torch.cuda.stream(self.copy_stream):
                dev[:ln].copy_(slot.t[:ln], non_blocking=True)
            self.copy_stream.synchronize()
            slot.release()
            self.q_ready.put((k, dev, None, ln, tail))

    def next(self):
        """-> (k, device buffer or None, pinned slot or None, length, tail)"""
        return self.flow.get(self.q_ready)

    def give_back(self, dev):
        self.dev_free.put(dev)

    def passthrough(self):
        self._through.set()

    def digest(self):
        return self.md5.digest()


class _Sink:
    """writes pieces to a file object in order from a writer thread, optionally hashing them in a second thread;
    device pieces are downloaded into a ring of pinned slots"""

    def __init__(self, flow, f, slot_bytes, hash_output=False):
        self.flow, self.f = flow, f
        self.md5 = hashlib.md5() if hash_output else None
        self.free = _ring(RING, slot_bytes)
        self.q_w, self.q_h = queue.Queue(), queue.Queue()
        self.written = 0
        first = len(flow.threads)
        flow.spawn(self._write)
        if self.md5 is not None:
            flow.spawn(self._hash)
        self.threads = flow.threads[first:]

    def _consume(self, q, use):
        while True:
            item = self.flow.get(q)
            if item is None:
                return
            view, rel = item
            use(view)
            if rel is not None:
                rel()

    def _write(self):
        self._consume(self.q_w, self.f.write)

    def _hash(self):
        self._consume(self.q_h, self.md5.update)

    def _put(self, view, slot=None):
        rel = None
        if slot is not None:
            slot.hold(2 if self.md5 is not None else 1)
            rel = slot.release
        self.written += len(view)
        self.q_w.put((view, rel))
        if self.md5 is not None:
            self.q_h.put((view, rel))

    def device(self, t):
        """download a device tensor (current stream) and queue it"""
        m = t.numel()
        if not m:
            return
        slot = self.flow.get(self.free).ensure(m)
        slot.t[:m].copy_(t)
        self._put(memoryview(slot.t.numpy())[:m], slot)

    def host(self, slot, m):
        """queue the first m bytes of a pinned _Slot (the caller still releases its own hold)"""
        if m:
            self._put(memoryview(slot.t.numpy())[:m], slot)

    def data(self, b):
        if len(b):
            self._put(memoryview(b))

    def zeros(self, m):
        while m > 0:
            k = min(m, _ZEROS.size)
            self._put(memoryview(_ZEROS)[:k])
            m -= k

    def finish(self):
        self.q_w.put(None)
        if self.md5 is not None:
            self.q_h.put(None)

    def digest(self):
        return self.md5.digest()


def _through(src, sink, dev, slot, m):
    """a window inside the raw tail: its input bytes go to the output as they are (a window uploaded before the
    source switched to pass-through is downloaded again)"""
    if dev is not None:
        sink.device(dev[:m])
        src.give_back(dev)
    else:
        sink.host(slot, m)
        slot.release()


def _run(work):
    """work(flow) with every thread joined before returning"""
    flow = _Flow()
    try:
        return work(flow)
    except _Stop:
        flow.check()
        raise
    finally:
        flow.close()


def window_parts(pk_len, raw_at, lo, hi, n, marker):
    """what a window [lo, hi) of an n-byte input contributes to the body, in order: ("body", a, b) = bytes of its
    own encoded packages, bytes objects, ("input", a, b) = its input bytes (offsets relative to lo).  pk_len = bytes of
    its packages before the rest of the file turns raw, raw_at = the input position where that happens inside this
    window (None if it does not).  A window behind raw_at contributes ("input", 0, hi - lo); the last window is
    followed by the END package (distributed.end_package).  A raw package of 4 GiB or more raises struct.error here,
    before any part of the window is written."""
    parts = [("body", 0, pk_len)]
    if raw_at is not None:
        parts += [D.raw_package_header(marker, n - raw_at), ("input", raw_at - lo, hi - lo)]
    return parts


def _emit(sink, parts, body, inp):
    for p in parts:
        if isinstance(p, bytes):
            sink.data(p)
        else:
            sink.device((body if p[0] == "body" else inp)[p[1]:p[2]])


class Counters:
    """what AdaptiveCompressor's chunk_stats are built from, summed window by window"""

    def __init__(self):
        self.n_packages = 0
        self.n_comp = 0
        self.usage = [0] * 5          # [raw, 1, 2, 3, 4]
        self.saved = 0                # sum of orig - comp - overhead over compressed packages
        self.payload = 0              # sum of comp over compressed packages

    def add_packages(self, packages, ovh):
        for t, orig, comp in packages:
            self.n_packages += 1
            if t == 255:
                self.usage[0] += 1
                continue
            self.n_comp += 1
            self.saved += orig - comp - ovh
            self.payload += comp
            if 1 <= t <= 4:
                self.usage[t] += 1


# ---- windows ---------------------------------------------------------------------------------------------------
def fixed_windows(n, chunk, W):
    """[(lo, hi)]: whole chunks, at least one per window"""
    step = max(1, int(W) // chunk) * chunk
    return [(lo, min(n, lo + step)) for lo in range(0, n, step)] or [(0, 0)]


def dyn_windows(n, candidates, W):
    """[(lo, hi)]: whole segments of 64 * g bytes (as dyn_shard_ranges), at least one per window"""
    seglen = D.DYN_SEGU * D._gcd_of(candidates)
    step = max(1, int(W) // seglen) * seglen
    return [(lo, min(n, lo + step)) for lo in range(0, n, step)] or [(0, 0)]


def body_windows(body_len, W):
    step = max(1, int(W))
    return [(lo, min(body_len, lo + step)) for lo in range(0, body_len, step)]


# ---- device memory of each driver (DESIGN.md §4.6): every buffer is a torch tensor --------------------------
def fixed_device_bytes(W, chunk, marker_bytes=4):
    """DEV_SLOTS input windows + the body bound + the workspace of one window of whole chunks"""
    lib = L.lib()
    w = max(1, int(W) // chunk) * chunk
    return DEV_SLOTS * w + int(lib.ambc_compress_bound(w, chunk, marker_bytes)) + int(lib.ambc_compress_workspace_bytes(w, chunk))


def dynamic_device_bytes(W, candidates, marker_bytes=4):
    """DEV_SLOTS input windows with their 8192-byte halo + the walk's workspace + the encoder's output bound"""
    cands = sorted({int(c) for c in candidates}, reverse=True)
    seglen = D.DYN_SEGU * D._gcd_of(cands)
    w = max(1, int(W) // seglen) * seglen
    ws = int(L.lib().ambc_dyn_range_workspace_bytes(0, w, w, (C.c_uint32 * len(cands))(*cands), len(cands)))
    return DEV_SLOTS * (w + D.DYN_HALO) + ws + _encode_bound(w, marker_bytes)


def _encode_bound(w, marker_bytes):
    return w + D.DYN_HALO + max(w // 256 + 2, 1) * (marker_bytes + 14) + 64  # as engine.dyn_range_encode


def decompress_device_bytes(W, budget, marker_bytes=4, n_cand=None, big=0):
    """DEV_SLOTS body windows with their header halo + the range index's workspace for n_cand marker candidates
    (by default its first guess; a body with more marker occurrences needs more) + the window's table + the output
    piece of `budget` bytes.  big = what the largest package adds: its payload behind a window's halo and the part of
    its output above the budget (0 for the chunk sizes compress writes; at most 2 * (2^32 - 1))"""
    span = int(W) + D.range_halo(marker_bytes)
    n_cand = int(W) // 2048 + 64 if n_cand is None else n_cand  # the index's first guess; it grows past it
    entries = span // (marker_bytes + 14) + int(W) // 65536 + 4
    return (DEV_SLOTS * span + int(L.lib().ambc_range_workspace_bytes(int(W), n_cand)) + 32 * entries + int(budget) +
            big)


# ---- compress --------------------------------------------------------------------------------------------------
def compress_fixed(path, f, n, chunk, W, mask=L.NATIVE_MASK, flags=0, marker=engine.FIXED_MARKER):
    """the fixed grid of `path` (n bytes) -> its body written to the file object f.  -> (body length, input MD5,
    Counters).  Raises struct.error before writing the raw package when it would be 4 GiB or more, as the in-memory
    path does (adaptive_compressor.py:617-619)."""
    lib = engine.require_cuda()
    mb = len(marker)
    ovh = mb + 14
    wins = fixed_windows(n, chunk, W)
    wmax = max(hi - lo for lo, hi in wins)
    out = torch.empty(int(lib.ambc_compress_bound(wmax, chunk, mb)), dtype=torch.uint8, device="cuda")
    work = torch.empty(max(int(lib.ambc_compress_workspace_bytes(wmax, chunk)), 1), dtype=torch.uint8, device="cuda")
    pcr = bool(flags & L.F_PER_CHUNK_RAW)
    cnt = Counters()

    def work_fn(flow):
        src = _Source(flow, path, [(lo, hi - lo, hi - lo) for lo, hi in wins], wmax, hash_input=True)
        sink = _Sink(flow, f, out.numel())
        raw = False
        for lo, hi in wins:
            _, dev, slot, m, _ = src.next()
            if raw:  # inside the raw tail: the input goes through from disk
                _through(src, sink, dev, slot, m)
                continue
            o = engine.compress_device(dev[:m], chunk, mask, flags, marker, out=out, work=work)
            nc = int(o.n_chunks)
            types = o.types.cpu().numpy()
            comps = o.comp_lens.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
            fr = int(o.first_raw) if not pcr else -1
            limit = fr if fr >= 0 else nc
            origs = np.full(limit, chunk, dtype=np.int64)
            if limit and limit == nc:
                origs[-1] = m - (limit - 1) * chunk
            t = types[:limit]
            cm = t != 255
            cnt.n_packages += int(o.n_packages)
            cnt.n_comp += int(cm.sum())
            cnt.usage[0] += int(limit - cm.sum()) + (1 if fr >= 0 else 0)
            for mid in (1, 2, 3, 4):
                cnt.usage[mid] += int((t == mid).sum())
            cnt.saved += int((origs[cm] - comps[:limit][cm] - ovh).sum())
            cnt.payload += int(comps[:limit][cm].sum())
            raw_at = lo + fr * chunk if fr >= 0 else None
            _emit(sink, window_parts(D.packed_bytes(int(o.body_len), m, fr, chunk, mb), raw_at, lo, hi, n, marker),
                  o.body, dev)
            if raw_at is not None:
                raw = True
                src.passthrough()
            src.give_back(dev)
        sink.data(D.end_package(marker))
        sink.finish()
        flow.join()
        return sink.written, src.digest(), cnt
    return _run(work_fn)


def compress_dynamic(path, f, n, candidates, W, mask=L.NATIVE_MASK, flags=0, marker=engine.FIXED_MARKER):
    """the multi-candidate mode over `path` (n bytes) -> its body written to f.  -> (body length, input MD5,
    Counters).  A raw package of 4 GiB or more raises AmbcError(E_ARG) before it is written, as in the
    in-memory path."""
    engine.require_cuda()
    mb = len(marker)
    ovh = mb + 14
    cands = sorted({int(c) for c in candidates}, reverse=True)
    wins = dyn_windows(n, cands, W)
    spans = [(lo, D.dyn_buffer_span(lo, hi, n)[1] - lo, hi - lo) for lo, hi in wins]
    smax = max(s[1] for s in spans)
    wmax = max(hi - lo for lo, hi in wins)
    out = torch.empty(_encode_bound(wmax, mb), dtype=torch.uint8, device="cuda")
    cnt = Counters()

    def work_fn(flow):
        src = _Source(flow, path, spans, smax, hash_input=True)
        sink = _Sink(flow, f, smax + 2 * 8192)
        e, stopped, work = 0, False, None
        for lo, hi in wins:
            _, dev, slot, m, _ = src.next()
            if stopped:
                _through(src, sink, dev, slot, hi - lo)
                continue
            buf = dev[:m]
            if e >= n or hi <= lo:
                src.give_back(dev)
                continue
            dr = engine.dyn_range_walk(buf, lo, hi, n, cands, mask, flags, mb, work=work)
            work = dr.work
            row = D.entry_row(dr.table, e, "the window at %d" % lo)
            if row[1] == L.DYN_UNRESOLVED:
                row = engine.dyn_range_resolve(dr, e)
            frag, stop, pk, _, _ = engine.dyn_range_encode(dr, e, marker, out=out)
            cnt.add_packages([(t, o, c) for _, t, o, c in pk], ovh)
            if stop is not None:
                D.refuse_dyn_raw(n, stop)
                cnt.add_packages([(255, n - stop, n - stop)], ovh)
            _emit(sink, window_parts(frag.numel(), stop, lo, hi, n, marker), frag, buf)
            if stop is not None:
                stopped = True
                src.passthrough()
            else:
                e = row[2]
            del dr
            src.give_back(dev)
        sink.data(D.end_package(marker))
        sink.finish()
        flow.join()
        return sink.written, src.digest(), cnt
    return _run(work_fn)


def find_marker(path, n, W, max_len=32, levels=(16, 24, 32)):
    """MarkerFinder.find_marker (marker_finder.py:22-123) over the windows of `path`: one pass per level tried,
    the L-bit windows of each file window flagged with the L - 1 bits before it as carry into one zeroed flag
    array.  -> (marker bytes, length in bits); ValueError when there is none."""
    lib = engine.require_cuda()
    wins = body_windows(n, W) or [(0, 0)]
    stream = engine._stream_ptr()
    end_window, total = b"", 0
    for lv in levels:
        Lb = min(lv, max_len)
        flags = torch.zeros(1 << Lb, dtype=torch.uint8, device="cuda")

        def work_fn(flow):
            src = _Source(flow, path, [(lo, hi - lo, 0) for lo, hi in wins], max(hi - lo for lo, hi in wins))
            window, before = b"", 0
            for _ in wins:
                _, dev, _, m, tail = src.next()
                carry, cb = D._bits_of(window, before, Lb - 1)
                L.check(lib.ambc_marker_flags_dev(C.c_void_p(dev.data_ptr() if m else 0), m, Lb, carry, cb,
                                                  C.c_void_p(flags.data_ptr()), stream))
                torch.cuda.current_stream().synchronize()
                _, (window, before) = D.carry_windows([before, m], [window, tail])
                src.give_back(dev)
            flow.join()
            return window, before
        end_window, total = _run(work_fn)
        tail, tail_bits = D._bits_of(end_window, total, 31)
        ln, val = C.c_uint32(0), C.c_uint64(0)
        rc = lib.ambc_marker_pick_dev(C.c_void_p(flags.data_ptr()), Lb, max_len, 8 * total, tail, tail_bits,
                                      C.byref(ln), C.byref(val), stream)
        del flags
        if rc == L.OK:
            return engine.marker_bytes(val.value, ln.value), ln.value
        if rc != L.E_NO_MARKER or Lb == max_len:
            L.check(rc)
    raise ValueError("Could not find a marker of length <= %d bits" % min(max_len, levels[-1]))


# ---- decompress ------------------------------------------------------------------------------------------------
def table_words(t_table, ne):
    """a table of ne 32-byte ambc_pkg entries as int64 words [src_off, dst_off, comp_len | orig_len << 32,
    type | out_len << 32] -> (words (a view: writing dst_off rewrites the table), output end of every entry).
    out_len is an unsigned 32-bit field: a raw tail or a type 5-7 package may claim 2^31 bytes or more."""
    w = t_table[:ne * 32].view(torch.int64).view(ne, 4)
    return w, w[:, 1] + ((w[:, 3] >> 32) & 0xFFFFFFFF)


def piece_cuts(dst, ends, budget):
    """cut a table whose entries write [dst[k], ends[k]) (ascending, dst[0] >= 0) into pieces of at most `budget`
    output bytes at entry boundaries; an entry larger than the budget is a piece of its own.  -> [(i, j, a, b)]:
    entries [i, j) write the output bytes [a, b), rebased to a; the first piece starts at 0."""
    ne = int(ends.numel())
    cuts, a, i = [], 0, 0
    last_end = int(ends[-1]) if ne else 0
    while i < ne:
        if last_end - a <= budget:
            j, b = ne, last_end
        else:
            j = max(int(torch.searchsorted(ends, torch.tensor([a + budget], device=ends.device), right=True)), i + 1)
            b = int(dst[j]) if j < ne else last_end
        cuts.append((i, j, a, b))
        a, i = b, j
    return cuts


def _decode_pieces(buf, t_table, ne, span, budget, km, sink, out, status):
    """decode one window's table into its output slice of `span` bytes, in the pieces of piece_cuts with each
    piece's dst_off rebased.  -> the device output buffer (grown when a piece needs it)"""
    a = 0
    if ne:
        w, ends = table_words(t_table, ne)
        for i, j, a, b in piece_cuts(w[:, 1], ends, budget):
            if a:
                w[i:j, 1] -= a
            if out.numel() < b - a:
                out = torch.empty(b - a, dtype=torch.uint8, device="cuda")
            piece, st = engine.range_decode(buf, t_table[i * 32:], j - i, b - a, km, out=out)
            status[0] += st[0]
            status[1] += st[1]
            sink.device(piece)
            a = b
    sink.zeros(span - a)
    return out


def decompress(path, f, header_size, body_len, orig_size, W, marker=engine.FIXED_MARKER, known_mask=L.NATIVE_MASK,
               out_budget=None):
    """decode the body of the .ambc file `path` (body_len bytes behind header_size) into f.  -> (output MD5,
    status [codec errors, length mismatches]).  Raises ValueError("Marker mismatch in chunk header.") where the
    serial walk would; f then holds part of the output."""
    engine.require_cuda()
    mb, km = len(marker), known_mask
    budget = int(out_budget or W)
    wins = body_windows(body_len, W)
    spans = [(header_size + lo, D.buffer_span(lo, hi, body_len, mb)[1] - lo, 0) for lo, hi in wins]
    smax = max([s[1] for s in spans] + [1])
    status = [0, 0]
    stage = []  # one pinned staging buffer of at most STAGE bytes for the payload bytes behind a halo

    def read_behind(fd, buf, at, off, need):
        if not stage:
            stage.append(torch.empty(min(need, STAGE), dtype=torch.uint8, pin_memory=True))
        st = stage[0]
        for p in range(0, need, st.numel()):
            k = min(st.numel(), need - p)
            _pread(fd, memoryview(st.numpy())[:k], off + p)
            buf[at + p:at + p + k].copy_(st[:k])

    def work_fn(flow):
        sink = _Sink(flow, f, budget, hash_output=True)
        src = _Source(flow, path, spans, smax) if wins else None
        state, o0, work, out = engine.range_init_state(), 0, None, torch.empty(budget, dtype=torch.uint8,
                                                                                  device="cuda")
        for k, (lo, hi) in enumerate(wins):
            _, dev, _, m, _ = src.next()
            ri = engine.range_index(dev[:m], lo, hi, body_len, orig_size, marker, km, work=work)
            work = ri.work
            exit_ = engine.range_fold(ri, state)
            if exit_.status == L.RANGE_MARKER:
                raise ValueError("Marker mismatch in chunk header.")  # adaptive_compressor.py:407
            done = exit_.status != L.RANGE_RUNNING and exit_.pkg_pos == L.RANGE_NO_PKG
            last = done or k == len(wins) - 1
            o1 = orig_size if last else engine.range_out_offset(exit_, hi, orig_size, mb, km)
            need = engine.range_table(ri, state, count_only=True)[4]
            buf = dev
            if need:  # payload bytes behind the halo, read into the same buffer
                if buf.numel() < m + need:
                    buf = torch.empty(m + need, dtype=torch.uint8, device="cuda")
                    buf[:m].copy_(dev[:m])
                read_behind(src.fd, buf, m, header_size + lo + m, need)
            t_table, ne, _, _, _ = engine.range_table(ri, state)
            out = _decode_pieces(buf, t_table, ne, o1 - o0, budget, km, sink, out, status)
            del ri, t_table
            src.give_back(buf)
            state, o0 = exit_, o1
            if done:
                break
        sink.zeros(orig_size - o0)
        sink.finish()
        # a walk that ended early leaves the reader waiting for slots: wait for the sink, close() ends the rest
        flow.join(sink.threads)
        return sink.digest(), status
    return _run(work_fn)

