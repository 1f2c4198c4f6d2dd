"""CompressionMethod plug-ins backed by the CUDA codecs (libambc.so).

Mirror of the reference's plug-in contract (compression_methods.py:7-67): property
`type_id`, `compress(data) -> bytes`, `decompress(data, original_length) -> bytes`,
`should_use(data, threshold=0.9) -> bool`, `calculate_overhead() -> int`.  Same bytes, same
exceptions (Huffman: ValueError for 256 distinct symbols, IndexError for one; :382, :527).
Each call is one batch-of-one kernel launch; the chunk path of AdaptiveCompressor does not go
through these objects (it runs the fused select kernel), they exist for API parity and for
per-codec tests.  Items are limited to 8192 bytes, the largest size any native method is
eligible for (adaptive_compressor.py:114-127)."""
from abc import ABC, abstractmethod

from . import _lib as L
from . import engine


class CompressionMethod(ABC):
    @property
    @abstractmethod
    def type_id(self):
        ...

    @abstractmethod
    def compress(self, data):
        ...

    @abstractmethod
    def decompress(self, data, original_length):
        ...

    def should_use(self, data, threshold=0.9):
        return True

    def calculate_overhead(self):
        return 0


def _raise_codec_error(code):
    if code == L.CODEC_INDEX_ERROR:
        raise IndexError("string index out of range")
    if code == L.CODEC_VALUE_ERROR:
        raise ValueError("byte must be in range(0, 256)")
    raise L.AmbcError(code, "codec failure")


class _NativeMethod(CompressionMethod):
    _id = 0

    @property
    def type_id(self):
        return self._id

    def compress(self, data):
        if not data:
            return b""
        out = engine.codec_encode_batch(self._id, [bytes(data)])[0]
        if isinstance(out, int):
            _raise_codec_error(out)
        return out

    def decompress(self, data, original_length):
        if not data:
            return b""
        out = engine.codec_decode_batch(self._id, [bytes(data)], [int(original_length)])[0]
        if isinstance(out, int):
            _raise_codec_error(out)
        return out

    def should_use(self, data, threshold=0.9):
        if not data:
            return False
        gates, _ = engine.should_use_batch([bytes(data)])
        return gates[0][self._id]


class RLECompression(_NativeMethod):
    """(byte, count) pairs, count <= 255 (compression_methods.py:70-180)"""
    _id = L.RLE


class DictionaryCompression(_NativeMethod):
    """greedy LZ77, window 4096, look-ahead 32, earliest-longest match (compression_methods.py:183-343)"""
    _id = L.DICT

    def __init__(self, window_size=4096, lookahead_size=32):
        if (window_size, lookahead_size) != (4096, 32):
            raise NotImplementedError("the CUDA Dictionary codec implements the reference's fixed window 4096 / look-ahead 32")
        self.window_size = window_size
        self.lookahead_size = lookahead_size


class HuffmanCompression(_NativeMethod):
    """table in first-occurrence order + MSB-first bit stream (compression_methods.py:346-574)"""
    _id = L.HUFFMAN


class DeltaCompression(_NativeMethod):
    """byte differences mod 256 (compression_methods.py:577-667)"""
    _id = L.DELTA


class DeflateCompression(CompressionMethod):
    """method id 5 (advanced_compression.py:71-107), where the reference calls zlib.  compress() writes a
    conforming zlib stream on the GPU (one fixed-Huffman block over a greedy LZ77 parse): stock
    zlib.decompress reads it, but it is not the byte string zlib.compress(level=9) would write, so this codec
    is reported separately and is not a candidate of the chunk trial.  decompress() inflates ANY zlib stream
    on the GPU with the reference's conventions: pad / truncate to original_length, and where zlib raises
    (bad header, invalid block, truncated stream, Adler-32 mismatch) original_length zero bytes."""

    @property
    def type_id(self):
        return L.DEFLATE

    def compress(self, data, level=9):
        if not data:
            return b""
        data = bytes(data)
        # items of the C-ABI are limited to 8192 bytes; longer inputs become several complete zlib streams only
        # in the sense of one stream per call, so they are refused rather than silently split
        out = engine.codec_encode_batch(L.DEFLATE, [data])[0]
        if isinstance(out, int):
            raise L.AmbcError(out, "DEFLATE encode failed")
        return out

    def decompress(self, data, original_length):
        if not data:
            return b""
        out = engine.codec_decode_batch(L.DEFLATE, [bytes(data)], [int(original_length)])[0]
        if isinstance(out, int):
            raise L.AmbcError(out, "DEFLATE decode failed")
        return out

    def should_use(self, data, threshold=0.9):
        """at least 64 bytes and an entropy below 8.0 (advanced_compression.py:99-107)"""
        if len(data) < 64:
            return False
        if len(data) > L.MAX_CODEC_CHUNK:
            return True  # (entropy 8.0 needs a perfectly flat histogram; the gate kernel takes items up to 8192 bytes)
        _, ent = engine.should_use_batch([bytes(data)])
        return not ent[0] >= 8.0


class _StdlibDecoder(CompressionMethod):
    """a codec the reference takes from the Python stdlib, decoded on the GPU only"""
    _id = 0
    _stock = ""

    @property
    def type_id(self):
        return self._id

    def compress(self, data):
        raise NotImplementedError("%s streams are decoded on the GPU but not written there: a GPU encoder's bytes "
                                  "would not be stock %s's, so they could not reproduce the reference's files"
                                  % (type(self).__name__, self._stock))

    def decompress(self, data, original_length):
        if not data:
            return b""
        out = engine.codec_decode_batch(self._id, [bytes(data)], [int(original_length)])[0]
        if isinstance(out, int):
            raise L.AmbcError(out, "%s decode failed" % type(self).__name__)
        return out

    def should_use(self, data, threshold=0.9):
        return False  # decode-only: never a candidate for compressing a chunk


class BZip2Compression(_StdlibDecoder):
    """method id 6, where the reference calls the stdlib's bz2.  decompress() has the semantics of
    bz2.decompress(data) -- BZh1..BZh9 streams, randomised blocks, concatenated streams, trailing bytes
    that do not start a stream ignored -- padded / truncated to original_length, and original_length zero
    bytes where bz2.decompress raises (bad data, CRC mismatch, truncated stream).  Decode only."""
    _id = L.BZIP2
    _stock = "libbzip2"


class LZMACompression(_StdlibDecoder):
    """method id 7, where the reference calls the stdlib's lzma.  decompress() has the semantics of
    lzma.decompress(data) with FORMAT_AUTO -- .xz streams with one LZMA2 filter and a None / CRC32 / CRC64
    check, stream padding, concatenated streams, the legacy .lzma header -- padded / truncated to
    original_length, and original_length zero bytes where lzma.decompress raises.  Other filter chains and the
    SHA-256 check are not implemented and count as errors.  Decode only."""
    _id = L.LZMA
    _stock = "liblzma"


class NoCompression(CompressionMethod):
    """identity (compression_methods.py:670-713)"""

    @property
    def type_id(self):
        return L.RAW

    def compress(self, data):
        return bytes(data)

    def decompress(self, data, original_length):
        if not data and original_length <= 0:
            return b""
        return engine.codec_decode_batch(L.RAW, [bytes(data)], [int(original_length)])[0]
