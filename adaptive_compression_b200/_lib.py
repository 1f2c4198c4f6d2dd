"""ctypes binding of libambc.so (include/ambc.h).  There is no CPU fallback: if the library
or a CUDA device is missing, every entry point raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AMBC_LIB_PATH") or os.path.join(_HERE, "libambc.so")  # env override: dev experiments only

OK, E_CUDA, E_ARG, E_CAPACITY, E_MARKER, E_TOO_LARGE, E_NO_MARKER = 0, -1, -2, -3, -4, -5, -6
RLE, DICT, HUFFMAN, DELTA, RAW = 1, 2, 3, 4, 255
DEFLATE = 5  # zlib streams (advanced_compression.py:71-107): a plug-in codec and a decodable package type, not a trial candidate
BZIP2, LZMA = 6, 7  # bz2 / lzma streams: decode-only plug-in codecs and decodable package types
NATIVE_MASK = (1 << 1) | (1 << 2) | (1 << 3) | (1 << 4)
MAX_CODEC_CHUNK = 8192
F_PER_CHUNK_RAW = 1
CODEC_INDEX_ERROR, CODEC_VALUE_ERROR = -1, -2


class AmbcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libambc error %d: %s" % (code, msg))
        self.code = code


class CompressResult(C.Structure):
    _fields_ = [("body_len", C.c_uint64), ("n_chunks", C.c_uint64), ("first_raw", C.c_int64),
                ("n_packages", C.c_uint64), ("map_type_off", C.c_uint64), ("map_comp_off", C.c_uint64),
                ("payload_bytes", C.c_uint64), ("usage", C.c_uint64 * 5)]


class ChunkInfo(C.Structure):
    _fields_ = [("pos", C.c_uint64), ("orig_len", C.c_uint32), ("comp_len", C.c_uint32), ("type", C.c_uint32),
                ("pad", C.c_uint32)]


class ShardRec(C.Structure):
    _fields_ = [("packed_bytes", C.c_uint64), ("first_raw", C.c_int64)]


class ShardSlot(C.Structure):
    _fields_ = [("offset", C.c_uint64), ("state", C.c_uint32), ("reserved", C.c_uint32)]


class Pkg(C.Structure):
    _fields_ = [("src_off", C.c_uint64), ("dst_off", C.c_uint64), ("comp_len", C.c_uint32),
                ("orig_len", C.c_uint32), ("type", C.c_uint32), ("out_len", C.c_uint32)]


class RangeState(C.Structure):
    """ambc_range_state: the walk's state handed from one body range to the next"""
    _fields_ = [("next_pos", C.c_uint64), ("out_before", C.c_uint64), ("pkg_pos", C.c_uint64), ("pkg_out", C.c_uint64),
                ("pkg_type", C.c_uint32), ("pkg_orig", C.c_uint32), ("pkg_comp", C.c_uint32), ("status", C.c_uint32)]


class Range(C.Structure):
    """ambc_range: what one rank holds after ambc_range_index"""
    _fields_ = [("lo", C.c_uint64), ("hi", C.c_uint64), ("body_len", C.c_uint64), ("orig_size", C.c_uint64),
                ("n_cand", C.c_uint64), ("work_bytes", C.c_uint64), ("work_dev", C.c_void_p),
                ("marker_bytes", C.c_uint32), ("known_mask", C.c_uint32), ("levels", C.c_uint32), ("reserved", C.c_uint32)]


class DynEntry(C.Structure):
    """ambc_dyn_entry: where the multi-candidate chain goes from one possible entry of a rank's input range"""
    _fields_ = [("entry", C.c_uint64), ("exit", C.c_uint64), ("stop", C.c_uint64), ("status", C.c_uint32),
                ("reserved", C.c_uint32)]


class DynRange(C.Structure):
    """ambc_dyn_range: what one rank holds after ambc_dyn_range_walk"""
    _fields_ = [("lo", C.c_uint64), ("hi", C.c_uint64), ("n", C.c_uint64), ("work_bytes", C.c_uint64),
                ("work_dev", C.c_void_p), ("host", C.c_void_p), ("n_entries", C.c_uint32), ("reserved", C.c_uint32)]


DYN_JOIN, DYN_LEAVE, DYN_STOP, DYN_UNRESOLVED = 0, 1, 2, 3
DYN_MAX_ENTRIES = 32
DYN_NONE = (1 << 64) - 1

RANGE_NO_PKG = (1 << 64) - 1
RANGE_RUNNING, RANGE_END, RANGE_TRUNCATED, RANGE_COMPLETE, RANGE_MARKER = 0, 1, 2, 3, 4

_lib = None

_SIGS = {
    "ambc_last_error": (C.c_char_p, []),
    "ambc_version": (C.c_int, []),
    "ambc_device_count": (C.c_int, []),
    "ambc_launch_count": (C.c_uint64, []),
    "ambc_compress_workspace_bytes": (C.c_uint64, [C.c_uint64, C.c_uint32]),
    "ambc_compress_bound": (C.c_uint64, [C.c_uint64, C.c_uint32, C.c_uint32]),
    "ambc_compress_dev": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_char_p,
                                    C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
                                    C.POINTER(CompressResult), C.c_void_p]),
    "ambc_compress_host": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_char_p,
                                     C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                     C.POINTER(CompressResult)]),
    "ambc_compress_dynamic_workspace_bytes": (C.c_uint64, [C.c_uint64, C.c_void_p, C.c_uint32]),
    "ambc_compress_dynamic_dev": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32,
                                            C.c_char_p, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
                                            C.POINTER(CompressResult), C.c_void_p, C.c_uint64, C.c_void_p]),
    "ambc_dyn_range_workspace_bytes": (C.c_uint64, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint32]),
    "ambc_dyn_range_walk": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint32,
                                      C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64, C.POINTER(DynRange),
                                      C.POINTER(DynEntry), C.c_uint32, C.POINTER(C.c_uint32), C.c_void_p]),
    "ambc_dyn_range_resolve": (C.c_int, [C.POINTER(DynRange), C.c_uint64, C.POINTER(DynEntry), C.c_void_p]),
    "ambc_dyn_range_encode": (C.c_int, [C.POINTER(DynRange), C.c_void_p, C.c_uint64, C.c_char_p, C.c_uint32, C.c_void_p,
                                        C.c_uint64, C.POINTER(CompressResult), C.c_void_p, C.c_uint64,
                                        C.POINTER(C.c_uint64), C.c_void_p]),
    "ambc_dyn_range_free": (None, [C.POINTER(DynRange)]),
    "ambc_index_host": (C.c_int, [C.c_void_p, C.c_uint64, C.c_char_p, C.c_uint32, C.c_uint64, C.c_uint32,
                                  C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "ambc_index_dev": (C.c_int, [C.c_void_p, C.c_uint64, C.c_char_p, C.c_uint32, C.c_uint64, C.c_uint32,
                                 C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_void_p]),
    "ambc_range_workspace_bytes": (C.c_uint64, [C.c_uint64, C.c_uint64]),
    "ambc_range_index": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_char_p, C.c_uint32,
                                   C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64, C.POINTER(Range), C.c_void_p]),
    "ambc_range_fold": (C.c_int, [C.POINTER(Range), C.POINTER(RangeState), C.POINTER(RangeState), C.c_void_p]),
    "ambc_range_table": (C.c_int, [C.POINTER(Range), C.POINTER(RangeState), C.c_void_p, C.c_uint64,
                                   C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                   C.POINTER(C.c_uint64), C.c_void_p]),
    "ambc_range_out_offset": (C.c_uint64, [C.POINTER(RangeState), C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]),
    "ambc_decompress_dev": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
                                      C.c_void_p, C.c_void_p]),
    "ambc_decompress_dev_mask": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
                                           C.c_uint32, C.c_void_p, C.c_void_p]),
    "ambc_decompress_host": (C.c_int, [C.c_void_p, C.c_uint64, C.c_char_p, C.c_uint32, C.c_uint32, C.c_void_p,
                                       C.c_uint64, C.c_void_p]),
    "ambc_codec_bound": (C.c_uint64, [C.c_int, C.c_uint32]),
    "ambc_codec_encode_batch": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64,
                                          C.c_void_p, C.c_void_p]),
    "ambc_codec_decode_batch": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                          C.c_uint64, C.c_void_p, C.c_void_p]),
    "ambc_should_use_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ambc_marker_flags_dev": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint64, C.c_uint32, C.c_void_p,
                                        C.c_void_p]),
    "ambc_marker_pick_dev": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint32,
                                       C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.c_void_p]),
    "ambc_find_marker_dev": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint32),
                                       C.POINTER(C.c_uint64), C.c_void_p]),
    "ambc_shard_place": (C.c_int, [C.POINTER(ShardRec), C.c_uint32, C.POINTER(C.c_uint64), C.c_uint32, C.c_uint32,
                                   C.POINTER(ShardSlot)]),
    "ambc_synth_dev": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p]),
    "ambc_enable_timing": (None, [C.c_int]),
    "ambc_last_timing": (C.c_int, [C.POINTER(C.c_float)]),
    "ambc_host_alloc": (C.c_void_p, [C.c_uint64]),
    "ambc_host_free": (None, [C.c_void_p]),
    # test hooks (include/ambc.h, last section)
    "ambc_set_walk_threads": (None, [C.c_uint64, C.c_uint]),
    "ambc_scan_state_bytes": (C.c_uint64, []),
}


def exported_symbols():
    """names include/ambc.h declares (used by the CPU-only load test)"""
    return sorted(_SIGS)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libambc.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "or `make -C adaptive_compression_b200/csrc`); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != OK:
        msg = lib().ambc_last_error().decode("utf-8", "replace")
        if rc == E_MARKER:
            raise ValueError("Marker mismatch in chunk header.")  # adaptive_compressor.py:407
        if rc == E_NO_MARKER:
            raise ValueError(msg)                                 # marker_finder.py:123
        raise AmbcError(rc, msg)
    return rc
