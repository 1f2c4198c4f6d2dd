"""AdaptiveCompressor: the reference's compress / decompress API (adaptive_compressor.py:49-700)
over the CUDA chunk path.

Byte compatibility follows the reference's CODE (SURVEY.md §0): constant 32-bit marker
FF FF 00 00 (:303-310), 47-byte header (:312-325), 18-byte package headers (:609-621), 16-byte
END package (:595-607), "rest of the file is one raw package" when a chunk has no winner
(:586-590), verbatim copy when header+body is larger than the input (:241-247).

What differs, on purpose:
  * CHUNK_SIZE_CANDIDATES defaults to the reference's own list 131072..1024 (:61-62), so a caller without
    arguments writes the files the reference writes (dynamic multi-size search, :548-584: every size is
    tried at every position on the GPU).  chunk_size=N selects ONE size -- the fixed grid of the benchmarked
    path (--chunk-size 4096 in BASELINE.json's configs), an order of magnitude faster.  Candidate lists are
    searched largest first (the reference honours the list order on ratio ties; its own list is descending).
  * only the repo-native methods 1-4 (+255) are loaded by default; DEFLATE (id 5), BZIP2 (id 6) and LZMA (id 7) on
    request (methods=[..., 5, 6, 7]): decoded on the GPU, not trial candidates; the other third-party codecs 8-11 are
    out of scope.
  * per_chunk_raw=True and use_marker_search=True are labelled extensions (files stay readable by
    the reference decoder)."""
import ctypes as C
import hashlib
import os
import secrets
import shutil
import stat
import struct
import threading
import time

import numpy as np
import torch

from . import _lib as L
from . import engine, windowed
from .compression_methods import (BZip2Compression, DeflateCompression, DeltaCompression, DictionaryCompression,
                                  HuffmanCompression, LZMACompression, NoCompression, RLECompression)
from .marker_finder import MarkerFinder

METHOD_NAMES = {1: "RLE", 2: "Dictionary", 3: "Huffman", 4: "Delta", 5: "DEFLATE", 6: "BZIP2", 7: "LZMA",
                8: "ZStandard", 9: "LZ4", 10: "Brotli", 11: "LZHAM", 255: "No Compression"}
METHOD_CHUNK_PREFS = {1: (32, 4096), 2: (128, 8192), 3: (32, 8192), 4: (32, 4096), 5: (64, 65536),
                      6: (1024, 262144), 7: (8192, 524288), 8: (512, 262144), 9: (1024, 65536),
                      10: (1024, 262144), 11: (1024, 262144), 255: (1, 999999999)}


REFERENCE_CANDIDATES = (131072, 65536, 32768, 16384, 8192, 4096, 2048, 1024)  # adaptive_compressor.py:61-62

WINDOW_CAP = 4 << 30      # largest window of the windowed path (DESIGN.md §4.6)
WINDOW_MIN = 16 << 20
MEMORY_MARGIN = 2 << 30   # device memory left free for the allocator's rounding, other streams and library scratch


def window_bytes(need, device_bytes):
    """The path of one compress / decompress call.  need = device bytes the in-memory path allocates for this file,
    device_bytes(W) = those of the windowed path with windows of W bytes.  -> None when `need` fits the free device
    memory with a margin (the in-memory path runs), else the window size: the largest power of two up to WINDOW_CAP
    whose windowed path fits."""
    free = torch.cuda.mem_get_info()[0] + torch.cuda.memory_reserved() - torch.cuda.memory_allocated()
    if need + MEMORY_MARGIN <= free:
        return None
    w = WINDOW_CAP
    while w > WINDOW_MIN and device_bytes(w) + MEMORY_MARGIN > free:
        w //= 2
    return w


def _temp_beside(path):
    """-> (temporary file, final file): an empty file beside the file `path` names (through a symlink, which is
    kept), with the mode of the file it will replace, or else the mode a new file gets there (0o666 less the
    umask, applied by open)"""
    target = os.path.realpath(path)
    try:
        mode = stat.S_IMODE(os.stat(target).st_mode)
    except FileNotFoundError:
        mode = None
    while True:
        tmp = os.path.join(os.path.dirname(target), ".%s.%s.tmp" % (os.path.basename(target), secrets.token_hex(6)))
        try:
            fd = os.open(tmp, os.O_WRONLY | os.O_CREAT | os.O_EXCL, 0o666)
            break
        except FileExistsError:
            continue
    try:
        if mode is not None:
            os.fchmod(fd, mode)
    finally:
        os.close(fd)
    return tmp, target


class AdaptiveCompressor:
    MAGIC_NUMBER = b"AMBC"
    FORMAT_VERSION = 2
    CHUNK_SIZE_CANDIDATES = list(REFERENCE_CANDIDATES)

    def __init__(self, marker_max_length=32, sample_size=10000, chunk_size=None, methods=None,
                 disable_methods=None, per_chunk_raw=False, use_marker_search=False):
        self.marker_finder = MarkerFinder(marker_max_length)
        self.sample_size = sample_size
        self.marker_bytes = None
        self.marker_length = 0
        self.marker_pattern = ""
        self.marker_bytes_aligned = b""
        self.marker_byte_length = 0
        self.use_multithreading = False
        self.max_workers = max(1, (os.cpu_count() or 2) - 1)
        self.progress_callback = None
        self.per_chunk_raw = bool(per_chunk_raw)
        self.use_marker_search = bool(use_marker_search)
        if chunk_size is not None:
            if isinstance(chunk_size, str):
                if chunk_size.lower() not in ("dynamic", "auto", "default"):
                    raise ValueError("chunk_size: an int, a list of candidate sizes, or 'dynamic'")
                chunk_size = REFERENCE_CANDIDATES
            if isinstance(chunk_size, (list, tuple)):
                self.CHUNK_SIZE_CANDIDATES = sorted({int(c) for c in chunk_size}, reverse=True)
            else:
                self.CHUNK_SIZE_CANDIDATES = [int(chunk_size)]
        self.compression_methods = [RLECompression(), DictionaryCompression(), HuffmanCompression(),
                                    DeltaCompression(), NoCompression()]
        if methods is not None:
            keep = set(int(m) for m in methods) | {255}
            # DEFLATE, BZIP2 and LZMA on request (the stdlib codecs of advanced_compression.py): packages of these
            # types decode on the GPU; the chunk trial of compress() stays with methods 1-4, see _method_mask
            self.compression_methods[4:4] = [cls() for mid, cls in ((5, DeflateCompression), (6, BZip2Compression),
                                                                     (7, LZMACompression)) if mid in keep]
            self.compression_methods = [m for m in self.compression_methods if m.type_id in keep]
        if disable_methods:
            drop = set(int(m) for m in disable_methods) - {255}
            self.compression_methods = [m for m in self.compression_methods if m.type_id not in drop]
        self.method_lookup = {m.type_id: m for m in self.compression_methods}
        self.method_names = dict(METHOD_NAMES)
        self.method_chunk_prefs = dict(METHOD_CHUNK_PREFS)
        self.chunk_stats = {}
        self.last_timing = {}
        self.last_status = [0, 0]  # decompress: [packages whose codec raised, packages with a length mismatch]

    # ---- no-op knobs kept for API compatibility (adaptive_compressor.py:179-194) ----
    def set_progress_callback(self, callback):
        self.progress_callback = callback

    def enable_multithreading(self, max_workers=None):
        self.use_multithreading = True
        if max_workers:
            self.max_workers = max_workers
        print(f"Multithreading enabled with {self.max_workers} workers")

    def disable_multithreading(self):
        self.use_multithreading = False
        print("Multithreading disabled")

    # ---- marker (adaptive_compressor.py:196-219, 303-310) ----
    def _init_marker(self, marker_bytes, marker_length):
        self.marker_bytes = bytes(marker_bytes)
        self.marker_length = marker_length
        nb = (marker_length + 7) // 8
        value = int.from_bytes(self.marker_bytes[:nb], "big") >> (8 * nb - marker_length) if marker_length else 0
        self.marker_pattern = format(value, "0%db" % marker_length) if marker_length else ""
        self.marker_bytes_aligned = (value << (8 * nb - marker_length)).to_bytes(nb, "big") if nb else b""
        self.marker_byte_length = nb

    def _find_marker(self, file_data, sample_size):
        if self.use_marker_search:
            return self.marker_finder.find_marker(file_data, None)
        return b"\xff\xff\x00\x00", 32

    # ---- header (adaptive_compressor.py:312-358) ----
    def _build_header(self, marker_bytes, marker_len, chksum, original_size, compressed_size=0):
        body = (bytes([marker_len]) + bytes(marker_bytes) + b"\x01" + chksum +
                struct.pack("<QQ", original_size, compressed_size))
        hsize = 4 + 1 + 4 + len(body)
        return self.MAGIC_NUMBER + bytes([self.FORMAT_VERSION]) + struct.pack("<I", hsize) + body

    def _parse_header(self, data):
        if data[:4] != self.MAGIC_NUMBER:
            raise ValueError("Magic mismatch")
        version = data[4]
        if version > self.FORMAT_VERSION:
            raise ValueError(f"Unsupported version: {version}")
        (hdr_size,) = struct.unpack("<I", data[5:9])
        marker_len = data[9]
        msize = (marker_len + 7) // 8
        ctype = data[10 + msize]
        csum_size = 16 if ctype == 1 else 0
        p = 11 + msize + csum_size
        orig_size, comp_size = struct.unpack("<QQ", data[p:p + 16])
        return {"format_version": version, "header_size": hdr_size, "marker_length": marker_len,
                "marker_bytes": bytes(data[10:10 + msize]), "checksum_type": ctype,
                "checksum": bytes(data[11 + msize:p]), "original_size": orig_size, "compressed_size": comp_size}

    # ---- configuration checks ----
    def _fixed_chunk(self):
        """the single candidate size, or None when several candidates are set (dynamic mode)"""
        c = list(self.CHUNK_SIZE_CANDIDATES)
        if not c or min(c) <= 0:
            raise ValueError("chunk size must be positive")
        if len(c) != 1:
            return None
        return int(c[0])

    def _method_mask(self):
        ids = [m.type_id for m in self.compression_methods if m.type_id != 255]
        foreign = [i for i in ids if i not in (1, 2, 3, 4, 5, 6, 7)]
        if foreign:
            raise NotImplementedError("only the repo-native methods 1-4 run on the B200 path; got %s" % foreign)
        if 5 in ids:
            # the GPU DEFLATE encoder does not write zlib.compress(level=9)'s bytes, so a trial with it could
            # not reproduce the reference's choices: it is a plug-in (DeflateCompression) and a decodable type
            print("DEFLATE (id 5) is decoded but takes no part in the chunk trial on the B200 path")
        for i in (6, 7):
            if i in ids:  # decode-only: there is no GPU encoder whose bytes would be libbzip2's / liblzma's
                print("%s (id %d) is decoded but takes no part in the chunk trial on the B200 path" % (METHOD_NAMES[i], i))
        return engine.method_mask([i for i in ids if i not in (5, 6, 7)])

    # ---- compress (adaptive_compressor.py:221-255) ----
    @staticmethod
    def _read_with_md5(path, slot):
        """file -> (pinned uint8 array, join() -> md5 digest): the file is read in pieces into page-locked memory
        while a thread hashes the pieces already there (MD5 is a serial chain at ~0.6 GB/s, the floor of this API;
        hashlib releases the GIL)"""
        n = os.path.getsize(path)
        buf = engine.pinned(slot, max(n, 1))
        h = hashlib.md5()
        done = [0]
        cv = threading.Condition()

        def hasher():
            pos = 0
            while pos < n:
                with cv:
                    while done[0] <= pos:
                        cv.wait()
                    upto = done[0]
                h.update(memoryview(buf)[pos:upto])
                pos = upto

        th = threading.Thread(target=hasher)
        th.start()
        piece = 32 << 20
        with open(path, "rb", buffering=0) as f:
            pos = 0
            while pos < n:
                got = f.readinto(memoryview(buf)[pos:min(n, pos + piece)])
                if not got:
                    raise IOError("short read of %s" % path)
                pos += got
                with cv:
                    done[0] = pos
                    cv.notify()

        def join():
            th.join()
            return h.digest()
        return buf[:n], join

    def _compress_need(self, n, chunk):
        """device bytes of the in-memory compress of n bytes, from the library's own size functions (marker of at
        most 4 bytes; the host-buffer path adds 1/8 to each cached buffer)"""
        lib = L.lib()
        if chunk is None:
            cands = sorted({int(c) for c in self.CHUNK_SIZE_CANDIDATES}, reverse=True)
            g = windowed.D._gcd_of(cands)
            need = 2 * n + (n // g + 3) * 18 + 80 + int(lib.ambc_compress_dynamic_workspace_bytes(
                n, (C.c_uint32 * len(cands))(*cands), len(cands)))
        else:
            need = (n + 64 + int(lib.ambc_compress_bound(n, chunk, 4)) + int(lib.ambc_compress_workspace_bytes(n, chunk)))
            need += need // 8
        if self.use_marker_search:  # the input, the 2^32 flags and the pick's scratch of the 32-bit level
            need = max(need, n + (2 << 32))
        return need

    def compress(self, input_file, output_file):
        start_t = time.time()
        engine.require_cuda()
        chunk = self._fixed_chunk()
        mask = self._method_mask()
        n = os.path.getsize(input_file)
        if chunk is None:
            W = window_bytes(self._compress_need(n, None),
                             lambda w: windowed.dynamic_device_bytes(w, self.CHUNK_SIZE_CANDIDATES))
        else:
            W = window_bytes(self._compress_need(n, chunk), lambda w: windowed.fixed_device_bytes(w, chunk))
        if W is not None:
            return self._compress_windowed(input_file, output_file, n, chunk, mask, W, start_t)
        file_data, md5_join = self._read_with_md5(input_file, "in")
        n = int(file_data.size)
        t_read = time.time()

        marker_bytes, marker_len = self._find_marker(file_data, self.sample_size)
        self._init_marker(marker_bytes, marker_len)
        flags = L.F_PER_CHUNK_RAW if self.per_chunk_raw else 0
        if chunk is None:  # several candidate sizes: the reference's dynamic mode (:548-584)
            t_in = torch.from_numpy(file_data).to("cuda") if n else torch.empty(0, dtype=torch.uint8, device="cuda")
            out = engine.compress_dynamic_device(t_in, self.CHUNK_SIZE_CANDIDATES, mask, flags, self.marker_bytes_aligned)
            self._fill_chunk_stats_packages(out.packages, n)
            body, body_len = None, int(out.body_len)
        else:
            # fixed grid: the pipelined host-buffer path of the C-ABI (ambc_compress_host)
            body, res, types, comps = engine.compress_host(file_data, n, chunk, mask, flags, self.marker_bytes_aligned)
            if res.first_raw >= 0 and not self.per_chunk_raw and n - res.first_raw * chunk > 0xFFFFFFFF:
                raise struct.error("'I' format requires 0 <= number <= 4294967295")  # as struct.pack at :617-619
            self._fill_chunk_stats(res, types, comps, n, chunk)
            body_len = int(res.body_len)
        t_gpu = time.time()
        header = self._build_header(marker_bytes[:self.marker_byte_length], marker_len, b"\0" * 16, n, body_len)
        final_size = len(header) + body_len
        if final_size > n:
            print("Compression bigger than original => store raw.")
            file_data.tofile(output_file)
            md5_join()
            stats = self._build_stats_raw(n, time.time() - start_t)
        else:
            if body is None:
                body = out.body.cpu().numpy()
            with open(output_file, "wb") as f:  # body first (the checksum is still being computed), header patched in
                f.write(header)
                body.tofile(f)
                header = self._build_header(marker_bytes[:self.marker_byte_length], marker_len, md5_join(), n, body_len)
                f.seek(0)
                f.write(header)
            stats = self._calculate_compression_stats(n, final_size, time.time() - start_t)
        self.last_timing = {"read_s": t_read - start_t, "gpu_s": t_gpu - t_read, "total_s": time.time() - start_t}
        return stats

    def _compress_windowed(self, input_file, output_file, n, chunk, mask, W, start_t):
        """compress() through windows of W bytes (windowed.py): the same file and stats; the output appears by a
        rename once complete"""
        if self.use_marker_search:
            marker_bytes, marker_len = windowed.find_marker(input_file, n, W, min(int(self.marker_finder.max_marker_length), 32))
        else:
            marker_bytes, marker_len = b"\xff\xff\x00\x00", 32
        self._init_marker(marker_bytes, marker_len)
        t_read = time.time()
        flags = L.F_PER_CHUNK_RAW if self.per_chunk_raw else 0
        tmp, target = _temp_beside(output_file)
        try:
            with open(tmp, "wb") as f:
                header = self._build_header(marker_bytes[:self.marker_byte_length], marker_len, b"\0" * 16, n, 0)
                f.write(header)
                if chunk is None:
                    body_len, md5, cnt = windowed.compress_dynamic(input_file, f, n, self.CHUNK_SIZE_CANDIDATES, W, mask,
                                                                   flags, self.marker_bytes_aligned)
                else:
                    body_len, md5, cnt = windowed.compress_fixed(input_file, f, n, chunk, W, mask, flags,
                                                                 self.marker_bytes_aligned)
                final_size = len(header) + body_len
                if final_size <= n:
                    f.seek(0)
                    f.write(self._build_header(marker_bytes[:self.marker_byte_length], marker_len, md5, n, body_len))
            t_gpu = time.time()
            self._store_chunk_stats(cnt.n_packages, cnt.n_comp, cnt.usage, cnt.saved, cnt.payload, n)
            if final_size > n:
                print("Compression bigger than original => store raw.")
                shutil.copyfile(input_file, tmp)
                stats = self._build_stats_raw(n, time.time() - start_t)
            else:
                stats = self._calculate_compression_stats(n, final_size, time.time() - start_t)
            os.replace(tmp, target)
        except BaseException:
            os.unlink(tmp)
            raise
        self.last_timing = {"read_s": t_read - start_t, "gpu_s": t_gpu - t_read, "total_s": time.time() - start_t}
        return stats

    def _store_chunk_stats(self, n_packages, n_comp, usage_counts, saved, payload, n):
        """chunk_stats as _init_stats/_update_stats (:457-480) leave them; usage_counts = [raw, 1, 2, 3, 4]"""
        ovh = self.marker_byte_length + 14
        usage = {m.type_id: 0 for m in self.compression_methods}
        for mid in (1, 2, 3, 4):
            if mid in usage:
                usage[mid] = int(usage_counts[mid])
        self.chunk_stats = {
            "total_chunks": int(n_packages), "compressed_chunks": int(n_comp), "raw_chunks": int(n_packages) - int(n_comp),
            "method_usage": usage, "bytes_saved": int(saved), "original_size": n,
            "compressed_size_without_overhead": int(payload), "overhead_bytes": ovh * int(n_comp) + self.marker_byte_length + 12,
        }

    def _fill_chunk_stats(self, out, types, comps, n, chunk):
        """same numbers as _init_stats/_update_stats (:457-480) + the END overhead (:393); out = CompressResult,
        types / comps = the per-chunk method map"""
        ovh = self.marker_byte_length + 14
        comps = comps.astype(np.int64)
        limit = int(out.n_chunks)
        if out.first_raw >= 0 and not self.per_chunk_raw:
            limit = int(out.first_raw)
        t = types[:limit]
        comp_mask = t != 255
        origs = np.full(limit, chunk, dtype=np.int64)
        if limit and limit == int(out.n_chunks):
            origs[-1] = n - (limit - 1) * chunk
        usage = {mid: int((t == mid).sum()) for mid in (1, 2, 3, 4)}
        self._store_chunk_stats(out.n_packages, int(comp_mask.sum()), [0] + [usage.get(mid, 0) for mid in (1, 2, 3, 4)],
                                (origs[comp_mask] - comps[:limit][comp_mask] - ovh).sum(),
                                comps[:limit][comp_mask].sum(), n)

    def _fill_chunk_stats_packages(self, packages, n):
        """_init_stats/_update_stats (:457-480) from a package list [(type, orig, comp)]"""
        cnt = windowed.Counters()
        cnt.add_packages(packages, self.marker_byte_length + 14)
        self._store_chunk_stats(cnt.n_packages, cnt.n_comp, cnt.usage, cnt.saved, cnt.payload, n)

    def _build_stats_raw(self, original_size, elapsed):
        tput = original_size / (1024 * 1024 * elapsed) if elapsed > 0 else 0.0
        chunk_stats = {"total_chunks": 1, "compressed_chunks": 0, "raw_chunks": 1, "method_usage": {},
                       "bytes_saved": 0, "original_size": original_size,
                       "compressed_size_without_overhead": original_size, "overhead_bytes": 0}
        return {"original_size": original_size, "compressed_size": original_size, "ratio": 1.0,
                "percent_reduction": 0.0, "elapsed_time": elapsed, "throughput_mb_per_sec": tput,
                "chunk_stats": chunk_stats, "overhead_bytes": 0, "compression_efficiency": 1.0}

    def _calculate_compression_stats(self, orig_size, comp_size, elapsed):
        if orig_size == 0:
            ratio, pr = 1.0, 0.0
        else:
            ratio = comp_size / orig_size
            pr = (1.0 - ratio) * 100.0
        throughput = orig_size / (1024 * 1024 * elapsed) if elapsed > 0 else 0.0
        eff = 1.0
        cs = self.chunk_stats
        if cs["compressed_chunks"] > 0:
            approx = 0
            for mid, cnt in cs["method_usage"].items():
                if mid != 255 and cnt > 0:
                    approx += (cnt / cs["total_chunks"]) * orig_size
            if approx > 0:
                eff = cs["compressed_size_without_overhead"] / approx
        return {"original_size": orig_size, "compressed_size": comp_size, "ratio": ratio, "percent_reduction": pr,
                "elapsed_time": elapsed, "throughput_mb_per_sec": throughput, "chunk_stats": cs,
                "overhead_bytes": cs.get("overhead_bytes", 0), "compression_efficiency": eff}

    # ---- decompress (adaptive_compressor.py:286-301) ----
    def decompress(self, input_file, output_file):
        start_t = time.time()
        engine.require_cuda()
        size = os.path.getsize(input_file)
        with open(input_file, "rb") as f:
            hdr = self._parse_header(f.read(64))
        body_len = max(size - hdr["header_size"], 0)
        # ambc_decompress_host caches the body, the output and a table ring, each with 1/8 on top
        need = (body_len + hdr["original_size"] + (4 << 20)) * 9 // 8
        # one package's payload behind a halo and its output piece may each reach 2^32 - 1 bytes
        W = window_bytes(need, lambda w: windowed.decompress_device_bytes(w, w, (hdr["marker_length"] + 7) // 8,
                                                                         big=2 * 0xFFFFFFFF))
        if W is not None:
            return self._decompress_windowed(input_file, output_file, size, hdr, W, start_t)
        cdata = engine.pinned("cin", max(size, 1))[:size]
        with open(input_file, "rb", buffering=0) as f:
            pos = 0
            while pos < size:
                got = f.readinto(memoryview(cdata)[pos:])
                if not got:
                    raise IOError("short read of %s" % input_file)
                pos += got
        hdr = self._parse_header(cdata[:64].tobytes())
        self._init_marker(hdr["marker_bytes"], hdr["marker_length"])
        body = cdata[hdr["header_size"]:]
        known = engine.method_mask([m.type_id for m in self.compression_methods if m.type_id != 255])
        # the pipelined host-buffer path of the C-ABI (ambc_decompress_host): the package walk on the host runs
        # ahead of the upload, decode and download overlap
        decompressed, status = engine.decompress_host(body, hdr["original_size"], self.marker_bytes_aligned, known)
        md5 = {}
        th = threading.Thread(target=lambda: md5.setdefault("d", hashlib.md5(decompressed).digest()))
        th.start()  # the checksum (a serial chain, GIL released) runs while the file is written
        decompressed.tofile(output_file)
        th.join()
        self.last_status = status
        if md5["d"] != hdr["checksum"]:  # (the output file stays, as in the reference: written at :294, checked at :297-299)
            raise ValueError("Checksum mismatch => possibly corrupted file.")
        if status != [0, 0]:  # cannot happen with a matching checksum unless the damage cancels out; say so anyway
            print("Warning: %d package(s) failed to decode, %d with a length mismatch" % (status[0], status[1]))
        elapsed = time.time() - start_t
        dsize = int(decompressed.size)
        return {"compressed_size": int(cdata.size), "decompressed_size": dsize, "elapsed_time": elapsed,
                "throughput_mb_per_sec": dsize / (1024 * 1024 * elapsed) if elapsed > 0 else 0.0}

    def _decompress_windowed(self, input_file, output_file, size, hdr, W, start_t):
        """decompress() through body windows of W bytes (windowed.py), the output bounded by W too.  Errors as in
        the reference: on a marker mismatch no output appears; on a checksum mismatch the output is written first"""
        self._init_marker(hdr["marker_bytes"], hdr["marker_length"])
        known = engine.method_mask([m.type_id for m in self.compression_methods if m.type_id != 255])
        orig = hdr["original_size"]
        tmp, target = _temp_beside(output_file)
        try:
            with open(tmp, "wb") as f:
                md5, status = windowed.decompress(input_file, f, hdr["header_size"], max(size - hdr["header_size"], 0),
                                                  orig, W, self.marker_bytes_aligned, known)
            os.replace(tmp, target)
        except BaseException:
            os.unlink(tmp)
            raise
        self.last_status = status
        if md5 != hdr["checksum"]:
            raise ValueError("Checksum mismatch => possibly corrupted file.")
        if status != [0, 0]:
            print("Warning: %d package(s) failed to decode, %d with a length mismatch" % (status[0], status[1]))
        elapsed = time.time() - start_t
        return {"compressed_size": size, "decompressed_size": orig, "elapsed_time": elapsed,
                "throughput_mb_per_sec": orig / (1024 * 1024 * elapsed) if elapsed > 0 else 0.0}
