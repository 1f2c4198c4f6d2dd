/*
 * include/ambc.h -- C ABI of libambc.so, the B200 (sm_100a) implementation of
 * adaptive-compression's chunked encode / select / decode hot path.
 *
 * This is the drop-in boundary: the reference is pure Python with no FFI of
 * its own, so these are the entry points a maintainer binds with ctypes from
 * adaptive_compressor.py / compression_methods.py / marker_finder.py (see
 * INTEGRATION.md for the stubs).  Each entry point cites the reference
 * function it replaces (file:line relative to the reference repo).
 *
 * Conventions
 *   - plain C symbols, plain pointers and sizes; no torch / C++ types.
 *   - return value: 0 = ok, <0 = error code below; text via ambc_last_error().
 *   - "_dev" pointers are CUDA device pointers owned by the caller (for
 *     example torch.empty(..., device="cuda").data_ptr()); `stream` is a
 *     cudaStream_t passed as void* (NULL = default stream).
 *   - there is NO CPU fallback: every call fails with AMBC_E_CUDA when no
 *     device / kernel image is available.
 */
#ifndef AMBC_H
#define AMBC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AMBC_OK 0
#define AMBC_E_CUDA (-1)      /* CUDA runtime error (no device, launch failure ...) */
#define AMBC_E_ARG (-2)       /* bad argument                                        */
#define AMBC_E_CAPACITY (-3)  /* output / workspace too small                        */
#define AMBC_E_MARKER (-4)    /* "Marker mismatch in chunk header."  (adaptive_compressor.py:406-407) */
#define AMBC_E_TOO_LARGE (-5) /* chunk larger than AMBC_MAX_CODEC_CHUNK for a codec call */
#define AMBC_E_NO_MARKER (-6) /* no absent bit string up to max length (marker_finder.py:123) */

/* method ids = package types (adaptive_compressor.py:97-110) */
#define AMBC_RLE 1
#define AMBC_DICT 2
#define AMBC_HUFFMAN 3
#define AMBC_DELTA 4
#define AMBC_DEFLATE 5 /* third-party codecs the reference loads from the Python stdlib: decoded only */
#define AMBC_BZIP2 6
#define AMBC_LZMA 7
#define AMBC_RAW 255
#define AMBC_METHOD_BIT(id) (1u << (id))
#define AMBC_NATIVE_MASK (AMBC_METHOD_BIT(1) | AMBC_METHOD_BIT(2) | AMBC_METHOD_BIT(3) | AMBC_METHOD_BIT(4))

/* largest chunk any native method is eligible for (adaptive_compressor.py:114-127) */
#define AMBC_MAX_CODEC_CHUNK 8192

/* flags of ambc_compress_* */
#define AMBC_F_PER_CHUNK_RAW 1u /* labelled extension: a losing chunk becomes its own type-255
                                   package instead of the reference's "rest of file raw" rule
                                   (adaptive_compressor.py:586-590).  Off = reference behaviour. */

/* codec result codes in out_len[] of the *_batch calls (the Python exception the
 * reference raises for that input) */
#define AMBC_CODEC_INDEX_ERROR (-1)
#define AMBC_CODEC_VALUE_ERROR (-2)

const char *ambc_last_error(void);
int ambc_version(void);
/* number of CUDA devices, or AMBC_E_CUDA */
int ambc_device_count(void);
/* kernels launched by this library since load (bench.py's gpu_launches) */
uint64_t ambc_launch_count(void);

/* ------------------------------------------------------------------ */
/* compress: AdaptiveCompressor._adaptive_compress                      */
/*   adaptive_compressor.py:363-394 (chunk loop), :537-590 (trial +      */
/*   argmin + rest-of-file-raw rule), :631-700 (re-compress + benefit    */
/*   check + framing), :595-621 (package / END framing)                  */
/* ------------------------------------------------------------------ */

typedef struct {
    uint64_t body_len;      /* bytes written to out (all packages + 16-byte END)            */
    uint64_t n_chunks;      /* grid chunks = ceil(n / chunk)                                 */
    int64_t first_raw;      /* first grid chunk with no winning method, -1 if none           */
    uint64_t n_packages;    /* data packages written                                         */
    uint64_t map_type_off;  /* byte offset in the workspace of uint8  type[n_chunks]         */
    uint64_t map_comp_off;  /* byte offset in the workspace of uint32 comp_len[n_chunks]     */
    uint64_t payload_bytes; /* sum of comp_len over compressed (non-raw) packages            */
    uint64_t usage[5];      /* packages per method id 1..4, [0] = raw packages               */
} ambc_compress_result;

/* bytes of device workspace ambc_compress_dev needs for an input of n bytes */
uint64_t ambc_compress_workspace_bytes(uint64_t n, uint32_t chunk);
/* upper bound of the body length (out_cap to allocate) */
uint64_t ambc_compress_bound(uint64_t n, uint32_t chunk, uint32_t marker_bytes);

/*
 * Device-resident input -> device-resident body (packages + END).  `chunk` is the
 * single CHUNK_SIZE_CANDIDATES entry (adaptive_compressor.py:61, :548).
 * `method_mask` = enabled method ids (AMBC_METHOD_BIT), trial order 1,2,3,4 as in
 * the reference's list (adaptive_compressor.py:131-134).  `marker` =
 * marker_bytes_aligned (adaptive_compressor.py:196-219), 1..4 bytes.
 * Synchronises `stream` before returning and fills *res.
 */
int ambc_compress_dev(const void *in_dev, uint64_t n, uint32_t chunk, uint32_t method_mask, uint32_t flags,
                      const uint8_t *marker, uint32_t marker_bytes, void *out_dev, uint64_t out_cap,
                      void *work_dev, uint64_t work_bytes, ambc_compress_result *res, void *stream);

/*
 * Same with HOST buffers (pinned memory recommended): H2D copy, kernels, D2H copy
 * of the body and of the per-chunk method map.  map_type / map_comp may be NULL.
 * Device buffers are cached inside the library between calls.
 */
int ambc_compress_host(const void *in_host, uint64_t n, uint32_t chunk, uint32_t method_mask, uint32_t flags,
                       const uint8_t *marker, uint32_t marker_bytes, void *out_host, uint64_t out_cap,
                       uint8_t *map_type, uint32_t *map_comp, ambc_compress_result *res);

/*
 * Multi-candidate ("dynamic chunk size") mode: the reference's default
 * CHUNK_SIZE_CANDIDATES = [131072 .. 1024] (adaptive_compressor.py:61-62) or any
 * strictly descending list whose gcd is a multiple of 16 and >= 256.  At every
 * position each candidate (clamped to the remaining bytes) is tried, the smallest
 * ratio (len + overhead) / size wins, larger candidates win ties
 * (adaptive_compressor.py:548-584); no winner -> the rest is one raw package.
 * map_out (optional, map_cap entries): the package list in file order.
 */
typedef struct {
    uint64_t pos;       /* offset of the chunk in the input */
    uint32_t orig_len;  /* chunk size                        */
    uint32_t comp_len;  /* payload bytes                     */
    uint32_t type;      /* package type                      */
    uint32_t pad;
} ambc_chunk_info;
uint64_t ambc_compress_dynamic_workspace_bytes(uint64_t n, const uint32_t *cands, uint32_t n_cands);
int ambc_compress_dynamic_dev(const void *in_dev, uint64_t n, const uint32_t *cands, uint32_t n_cands,
                              uint32_t method_mask, uint32_t flags, const uint8_t *marker, uint32_t marker_bytes,
                              void *out_dev, uint64_t out_cap, void *work_dev, uint64_t work_bytes,
                              ambc_compress_result *res, ambc_chunk_info *map_out, uint64_t map_cap, void *stream);

/*
 * The multi-candidate mode across ranks: every rank holds one input range [lo, hi) and walks its chain; the fold of
 * the ranks' entry tables is host arithmetic (adaptive_compression_b200/distributed.py).  lo and hi are multiples of
 * 64 * g (g = gcd of the candidates), except that the last rank's hi is n.  The chain enters a range at a multiple of
 * g in [lo, lo + min(8192, cands[0])): a non-raw package is at most that long.
 *
 *   1. ambc_dyn_range_walk    (no communication) walks the range's segments, stitches the chain from lo, and in the
 *      first re-entry launch walks every other possible entry lo + k * g until it meets the chain from lo in the
 *      range's first segment.  Fills one ambc_dyn_entry per possible entry (lo first).
 *   2. ambc_dyn_range_resolve runs more stitch rounds from an entry the walk left AMBC_DYN_UNRESOLVED, until the
 *      chain from it leaves the range or stops.
 *   3. ambc_dyn_range_encode  encodes and frames the rank's packages of the chain from its true entry with the
 *      records already walked: no raw tail, no END; map positions are global.  *stop = the position the chain
 *      stops at (the rest of the file is one raw package), ~0 if it leaves the range.
 *
 * buf_dev holds input bytes [lo, min(n, hi + 8192)), 16-byte aligned, and stays valid until the last call; the
 * host side of the walk lives in r->host until ambc_dyn_range_free.
 */
typedef struct {
    uint64_t entry;    /* input position the chain enters the range at                                       */
    uint64_t exit;     /* first position of the chain at or past hi (>= n: the chain is complete), ~0 if none */
    uint64_t stop;     /* strict mode: no winner there, the rest of the file is raw; ~0 if none              */
    uint32_t status;   /* AMBC_DYN_*                                                                          */
    uint32_t reserved;
} ambc_dyn_entry;
#define AMBC_DYN_JOIN 0       /* meets the chain from lo: exit / stop are that chain's                           */
#define AMBC_DYN_LEAVE 1      /* leaves the range at exit without meeting it                                     */
#define AMBC_DYN_STOP 2       /* stops at stop without meeting it                                                */
#define AMBC_DYN_UNRESOLVED 3 /* left the first segment at exit without meeting it: ambc_dyn_range_resolve       */
#define AMBC_DYN_MAX_ENTRIES 32

typedef struct {
    uint64_t lo, hi, n;   /* the rank's input range and the input length                                      */
    uint64_t work_bytes;  /* device workspace the range needs (also set when AMBC_E_CAPACITY is returned)     */
    void *work_dev;
    void *host;           /* the walk's records on the host (ambc_dyn_range_free)                             */
    uint32_t n_entries, reserved;
} ambc_dyn_range;

uint64_t ambc_dyn_range_workspace_bytes(uint64_t lo, uint64_t hi, uint64_t n, const uint32_t *cands, uint32_t n_cands);
/* Phase 1 (synchronises `stream`); tab gets r->n_entries <= AMBC_DYN_MAX_ENTRIES entries (cap of them at most) */
int ambc_dyn_range_walk(const void *buf_dev, uint64_t buf_len, uint64_t lo, uint64_t hi, uint64_t n,
                        const uint32_t *cands, uint32_t n_cands, uint32_t method_mask, uint32_t flags,
                        uint32_t marker_bytes, void *work_dev, uint64_t work_bytes, ambc_dyn_range *r,
                        ambc_dyn_entry *tab, uint32_t cap, uint32_t *n_tab, void *stream);
/* Phase 2: *out = the entry's row, resolved (a no-op for an entry the walk resolved).  Synchronises `stream`. */
int ambc_dyn_range_resolve(ambc_dyn_range *r, uint64_t entry, ambc_dyn_entry *out, void *stream);
/* Phase 3: the rank's packages into out_dev (res->body_len bytes); entry >= hi: none.  Synchronises `stream`. */
int ambc_dyn_range_encode(ambc_dyn_range *r, const void *buf_dev, uint64_t entry, const uint8_t *marker,
                          uint32_t marker_bytes, void *out_dev, uint64_t out_cap, ambc_compress_result *res,
                          ambc_chunk_info *map_out, uint64_t map_cap, uint64_t *stop, void *stream);
void ambc_dyn_range_free(ambc_dyn_range *r);

/* ------------------------------------------------------------------ */
/* decompress: AdaptiveCompressor._adaptive_decompress                  */
/*   adaptive_compressor.py:396-454                                     */
/* ------------------------------------------------------------------ */

typedef struct {
    uint64_t src_off;  /* payload offset in the body                      */
    uint64_t dst_off;  /* output offset                                   */
    uint32_t comp_len; /* payload bytes                                   */
    uint32_t orig_len; /* original_length field of the package header     */
    uint32_t type;     /* package type; AMBC_RAW also for unknown types   */
    uint32_t out_len;  /* bytes this entry contributes to the output      */
} ambc_pkg;

/*
 * Walk the package chain on the host (adaptive_compressor.py:399-430 and the stop
 * rule :444-445): validates markers, stops at END / truncated header / truncated
 * payload.  Raw packages are split into entries of at most 64 KiB.  `known_mask`
 * = method ids present in method_lookup (others are copied through, :432-435):
 * bits 1-4 the native methods, bit 5 DEFLATE, bit 6 BZIP2, bit 7 LZMA.
 * Pass table=NULL to count entries.  Returns AMBC_E_MARKER on a marker mismatch.
 */
int ambc_index_host(const uint8_t *body, uint64_t body_len, const uint8_t *marker, uint32_t marker_bytes,
                    uint64_t orig_size, uint32_t known_mask, ambc_pkg *table, uint64_t table_cap,
                    uint64_t *n_entries, uint64_t *out_bytes);

/*
 * The same table built on the GPU from a device-resident body (no host copy of the body needed):
 * marker scan, header parse, successor links, pointer jumping from position 0, placement scans.
 * Only positions reachable from position 0 become packages, exactly as in the serial walk; a marker
 * mismatch the walk would hit returns AMBC_E_MARKER.  table_dev may be NULL to obtain *n_entries
 * first.  Synchronises `stream`.
 */
int ambc_index_dev(const void *body_dev, uint64_t body_len, const uint8_t *marker, uint32_t marker_bytes,
                   uint64_t orig_size, uint32_t known_mask, ambc_pkg *table_dev, uint64_t table_cap,
                   uint64_t *n_entries, uint64_t *out_bytes, void *stream);

/*
 * Range-local index: the same walk (adaptive_compressor.py:396-454) split across ranks that each
 * hold one byte range [lo, hi) of the body, so that every GPU indexes and decodes its own range.
 *
 *   1. ambc_range_index  (no communication) finds the header candidates in [lo, hi) of the rank's
 *      buffer, parses them, links every candidate to its successor and builds jump and output-sum
 *      tables.  A successor at or beyond hi is an exit of the range.
 *   2. ambc_range_fold   runs once per rank in rank order on the state the previous rank returned
 *      (the first rank starts from AMBC_RANGE_INIT): a rank whose range holds the next header walks
 *      its chain to the exit or to the walk's end, every other rank passes the state on unchanged.
 *   3. ambc_range_table  lists the rank's part of the walk from its entry state (the state the fold
 *      handed to it) as ambc_pkg entries for ambc_decompress_dev_mask: src_off relative to the rank's
 *      buffer (= body position - lo), dst_off relative to out_lo.
 *
 * Ownership: a decoded package belongs to the rank that holds its header; a copied-through payload
 * (type 255 and types without a known_mask bit) belongs to whoever holds its bytes, in 64 KiB pieces,
 * and the zero pad behind it to the rank holding its last payload byte; the zero tail
 * [covered, orig_size) belongs to the last rank.  Rank r's output slice is [out_lo_r, out_lo_{r+1})
 * with out_lo_R = orig_size; decode it with ambc_decompress_dev_mask(orig_size = slice length).
 */
typedef struct {
    uint64_t next_pos;   /* body position of the next header on the chain                               */
    uint64_t out_before; /* output bytes of the walk before it (>= orig_size once complete)           */
    uint64_t pkg_pos;    /* header position of the package whose payload runs past the range that      */
                         /* listed it, AMBC_RANGE_NO_PKG if none                                         */
    uint64_t pkg_out;    /* its output offset                                                         */
    uint32_t pkg_type, pkg_orig, pkg_comp;
    uint32_t status;     /* AMBC_RANGE_*                                                              */
} ambc_range_state;
#define AMBC_RANGE_NO_PKG (~0ull)
#define AMBC_RANGE_RUNNING 0   /* the walk continues at next_pos                                        */
#define AMBC_RANGE_END 1       /* END package (:422-424)                                                */
#define AMBC_RANGE_TRUNCATED 2 /* out of body: header or payload cut off, or the body's end (:400-403, :425-427) */
#define AMBC_RANGE_COMPLETE 3  /* output complete (:444-445)                                            */
#define AMBC_RANGE_MARKER 4    /* "Marker mismatch in chunk header." (:405-407)                          */
#define AMBC_RANGE_INIT {0, 0, AMBC_RANGE_NO_PKG, 0, 0, 0, 0, AMBC_RANGE_RUNNING}

/* what one rank holds; ambc_range_index fills it, the later calls read it */
typedef struct {
    uint64_t lo, hi;        /* body range of this rank                                                 */
    uint64_t body_len;      /* length of the whole body                                                */
    uint64_t orig_size;
    uint64_t n_cand;        /* header candidates (marker occurrences) starting in [lo, hi)             */
    uint64_t work_bytes;    /* workspace this range needs (also set when AMBC_E_CAPACITY is returned)  */
    void *work_dev;
    uint32_t marker_bytes, known_mask, levels, reserved;
} ambc_range;

/* device workspace for a range of range_len bytes with n_cand candidates */
uint64_t ambc_range_workspace_bytes(uint64_t range_len, uint64_t n_cand);
/*
 * Phase 1.  buf_dev holds body[lo, lo + buf_len) with buf_len >= min(hi + marker_bytes + 13, body_len) - lo
 * (the range plus the header halo behind hi).  Counts the candidates first; when work_bytes is too
 * small returns AMBC_E_CAPACITY with r->n_cand and r->work_bytes set (allocate and call again).  The
 * tables stay in work_dev for the other calls; the buffer is not read again.  Synchronises `stream`.
 */
int ambc_range_index(const void *buf_dev, uint64_t buf_len, uint64_t lo, uint64_t hi, uint64_t body_len,
                     const uint8_t *marker, uint32_t marker_bytes, uint64_t orig_size, uint32_t known_mask,
                     void *work_dev, uint64_t work_bytes, ambc_range *r, void *stream);
/* Phase 2, one fold step: *out = the walk's state behind this range given *in (host structs).
 * Synchronises `stream`. */
int ambc_range_fold(const ambc_range *r, const ambc_range_state *in, ambc_range_state *out, void *stream);
/*
 * Phase 3: the rank's table from its entry state (table_dev NULL: count only).  *out_lo / *out_hi =
 * output offsets of its first and behind its last entry (out_hi excludes the zero tail);
 * *need = payload bytes a decoded package of this range needs beyond body position
 * min(hi + marker_bytes + 13, body_len): the buffer must hold them before decoding.  Synchronises `stream`.
 */
int ambc_range_table(const ambc_range *r, const ambc_range_state *entry, ambc_pkg *table_dev, uint64_t table_cap,
                     uint64_t *n_entries, uint64_t *out_lo, uint64_t *out_hi, uint64_t *need, void *stream);
/* output offset of the first byte a range starting at body position `lo` owns, given the state the
 * fold handed to it (pure host arithmetic) */
uint64_t ambc_range_out_offset(const ambc_range_state *s, uint64_t lo, uint64_t orig_size, uint32_t marker_bytes,
                               uint32_t known_mask);

/*
 * Decode every table entry into out_dev (orig_size bytes; zero padded / truncated
 * as adaptive_compressor.py:447-452).  status_dev (optional, uint32[2]):
 * [0] = entries whose codec raised (output zero-filled, :440-442),
 * [1] = entries whose decoded length differed from the package's nominal length (malformed
 *       stream; nominal: orig_len, min(comp_len, orig_len) for Delta, 0 for an empty payload).
 * Entries of types 6 (BZIP2) and 7 (LZMA) are left to ambc_decompress_dev_mask.
 */
int ambc_decompress_dev(const void *body_dev, uint64_t body_len, const ambc_pkg *table_dev, uint64_t n_entries,
                        void *out_dev, uint64_t orig_size, uint32_t *status_dev, void *stream);
/*
 * The same, and entries of types 6 / 7 are decoded when known_mask has bit 6 / 7 (pass the
 * known_mask the table was built with).  Without those bits it is ambc_decompress_dev: the same
 * kernels, launches and device memory.  The first call with bit 6 allocates 1 GiB of bzip2 block
 * scratch on the device, kept for later calls.
 */
int ambc_decompress_dev_mask(const void *body_dev, uint64_t body_len, const ambc_pkg *table_dev, uint64_t n_entries,
                             void *out_dev, uint64_t orig_size, uint32_t known_mask, uint32_t *status_dev,
                             void *stream);

/* host buffers: index walk + H2D + kernels + D2H.  status (optional) as above.  Packages of
 * every type whose bit is in known_mask are decoded, 6 and 7 included. */
int ambc_decompress_host(const void *body_host, uint64_t body_len, const uint8_t *marker, uint32_t marker_bytes,
                         uint32_t known_mask, void *out_host, uint64_t orig_size, uint32_t *status);

/* ------------------------------------------------------------------ */
/* codec plug-ins: CompressionMethod.compress / decompress / should_use */
/*   compression_methods.py:78-180 (RLE), :195-343 (Dictionary),         */
/*   :354-574 (Huffman), :585-667 (Delta), :678-713 (NoCompression);     */
/*   method 5 = DeflateCompression, advanced_compression.py:71-107, where */
/*   the reference calls zlib: encode writes a conforming zlib stream     */
/*   (RFC 1950 / 1951, one fixed-Huffman block) that stock zlib reads --  */
/*   not zlib.compress(level=9)'s own bytes, hence a plug-in reported     */
/*   separately and no candidate of the chunk trial; decode inflates any  */
/*   zlib stream, pads / truncates to original_length, and returns        */
/*   original_length zero bytes where zlib.decompress raises (:93-97).    */
/*   known_mask bit 5 makes packages of type 5 decodable in a body.       */
/*   methods 6 = BZip2Compression and 7 = LZMACompression, where the      */
/*   reference calls the stdlib's bz2 / lzma: decode only, with the       */
/*   semantics of bz2.decompress / lzma.decompress (FORMAT_AUTO: .xz     */
/*   with a lone LZMA2 filter and a None / CRC32 / CRC64 check, or the    */
/*   legacy .lzma header; concatenated streams, trailing bytes as the     */
/*   stdlib treats them); pad / truncate to original_length, zeros where  */
/*   the stdlib raises.  No encoder: its bytes would not be libbzip2's or */
/*   liblzma's.  known_mask bits 6 / 7 make such packages decodable.      */
/* ------------------------------------------------------------------ */

/*
 * Item i = in_dev[in_off[i] .. in_off[i+1]) (at most AMBC_MAX_CODEC_CHUNK bytes).
 * Payload i is written at out_dev + i*out_stride; out_len[i] = payload length or
 * AMBC_CODEC_*_ERROR.  out_stride must be >= ambc_codec_bound(method, max item).
 */
uint64_t ambc_codec_bound(int method, uint32_t n);
int ambc_codec_encode_batch(int method, const void *in_dev, const uint64_t *in_off_dev, uint32_t n_items,
                            void *out_dev, uint64_t out_stride, int32_t *out_len_dev, void *stream);
/*
 * Item i = payload in_dev[in_off[i] .. in_off[i+1]) with original_length
 * orig_len[i]; decoded bytes at out_dev + i*out_stride, out_len[i] = number of
 * bytes the reference's decompress() returns, or AMBC_CODEC_INDEX_ERROR.
 * Methods 5-7 take payloads and original lengths of any size the stride holds.
 * Method 7 uses the whole stride as its dictionary: a stream that decodes past
 * out_stride bytes gets out_len[i] = AMBC_E_CAPACITY (call again with a larger
 * stride; the bytes behind original_length must be decoded to verify the check).
 * Method 6 verifies every CRC whatever the stride.
 */
int ambc_codec_decode_batch(int method, const void *in_dev, const uint64_t *in_off_dev,
                            const uint32_t *orig_len_dev, uint32_t n_items, void *out_dev, uint64_t out_stride,
                            int32_t *out_len_dev, void *stream);
/*
 * should_use of all four methods: gates[i] bit (id) set when method id's gate is
 * true; entropy_dev (optional) receives the fp64 entropy of
 * compression_methods.py:566-574.
 */
int ambc_should_use_batch(const void *in_dev, const uint64_t *in_off_dev, uint32_t n_items, uint8_t *gates_dev,
                          double *entropy_dev, void *stream);

/* ------------------------------------------------------------------ */
/* marker search: MarkerFinder.find_marker  (marker_finder.py:22-123)   */
/* ------------------------------------------------------------------ */

/*
 * Presence flags of all L-bit windows of the MSB-first bit stream of
 * in_dev[0..n): flags_dev[v] = 1 when value v occurs.  flags_dev holds 2^L bytes
 * and must be zeroed by the caller (so that several shards / GPUs can be merged
 * with a byte-wise max all-reduce before ambc_marker_pick).  `carry` = the
 * (L-1) bits that precede this shard in the global stream (low bits, MSB first),
 * carry_bits = how many of them exist (0 for the first shard).
 */
int ambc_marker_flags_dev(const void *in_dev, uint64_t n, uint32_t L, uint64_t carry, uint32_t carry_bits,
                          uint8_t *flags_dev, void *stream);
/*
 * From the flags of length L derive every shorter length (a shorter value is
 * present iff it prefixes a present L-bit value or equals the stream's last
 * window, given by `tail` / tail_bits = the last min(L-1, nbits) bits of the whole
 * stream) and return the smallest length in [1, min(L, max_len)] with an absent
 * value: *out_len bits, *out_value the smallest absent value.  AMBC_E_NO_MARKER
 * when every value up to min(L, max_len) is present.  total_bits = bits of the
 * whole stream.
 */
int ambc_marker_pick_dev(const uint8_t *flags_dev, uint32_t L, uint32_t max_len, uint64_t total_bits,
                         uint64_t tail, uint32_t tail_bits, uint32_t *out_len, uint64_t *out_value, void *stream);
/* single-GPU convenience: device input -> (marker value, length) */
int ambc_find_marker_dev(const void *in_dev, uint64_t n, uint32_t max_len, uint32_t *out_len, uint64_t *out_value,
                         void *stream);

/* ------------------------------------------------------------------ */
/* synthetic corpus (bench / tests): counter-based, any byte range       */
/* ------------------------------------------------------------------ */
/* fills out_dev[0..n) with bytes [offset, offset+n) of corpus (seed, kind_mask) */
int ambc_synth_dev(void *out_dev, uint64_t offset, uint64_t n, uint64_t seed, uint32_t kind_mask, void *stream);

/* ------------------------------------------------------------------ */
/* measurement support (bench.py): per-kernel device times              */
/* ------------------------------------------------------------------ */
/* when enabled, ambc_compress_dev / ambc_decompress_dev bracket their kernels with CUDA events
 * on the caller's stream; ambc_last_timing returns the most recent call's milliseconds:
 * ms[0] k_select, ms[1] size scan (3 small kernels), ms[2] k_pack, ms[3] k_decode (+tail zero). */
void ambc_enable_timing(int on);
int ambc_last_timing(float *ms4);

/* ---- multi-GPU placement (SURVEY.md 8e) ------------------------------------------------------------
 * Shards are contiguous chunk ranges compressed independently ("as if no earlier shard had hit a chunk
 * without a winner").  Every rank all-gathers one 16-byte record (the only exchange of the data path;
 * torch.distributed / NCCL moves it, this call folds it): packed_bytes = bytes of its local body before
 * its first raw chunk (END and local raw package removed), first_raw = GLOBAL index of its first chunk
 * without a winner or -1.  The fold applies the rest-of-file-raw rule (adaptive_compressor.py:586-590)
 * across shards: out[r].offset = byte offset of rank r's contribution in the global body and
 * out[r].state = AMBC_SHARD_PACKED (its packed fragment), AMBC_SHARD_RAW_STARTS (packed part, then the
 * header of the one global raw package and its input from the raw chunk on) or AMBC_SHARD_IN_RAW_TAIL
 * (its input bytes, verbatim, inside that package).  first_byte[r] = input byte offset of rank r's shard
 * (a multiple of the chunk size, or the input length for an empty trailing rank -- byte offsets rather than
 * chunk indices so that such a rank lands at the end of the raw data when the last chunk is partial).
 * Pure host arithmetic; needs no device. */
typedef struct { uint64_t packed_bytes; int64_t first_raw; } ambc_shard_rec;
typedef struct { uint64_t offset; uint32_t state; uint32_t reserved; } ambc_shard_slot;
#define AMBC_SHARD_PACKED 0
#define AMBC_SHARD_RAW_STARTS 1
#define AMBC_SHARD_IN_RAW_TAIL 2
int ambc_shard_place(const ambc_shard_rec *recs, uint32_t n_ranks, const uint64_t *first_byte, uint32_t chunk,
                     uint32_t marker_bytes, ambc_shard_slot *out);

/* ---- threading ----------------------------------------------------------------------------------------
 * The *_host calls serialise on a library mutex.  The *_dev calls keep per-DEVICE scratch (side stream and
 * events of the decoders, index scratch, kernel timers): call them from ONE host thread per device at a
 * time (different devices may be driven concurrently, one thread each). */

/* ---- test hooks (exported, not part of the reference-facing surface) ----------------------------------
 * ambc_set_walk_threads lets small bodies exercise the helper threads of ambc_index_host (min_bytes = body size
 * from which helpers start, threads = 0 for the host cores divided by LOCAL_WORLD_SIZE, at most 8);
 * ambc_scan_state_bytes = size of the per-piece state record ambc_compress_host downloads.  None of them changes
 * any result. */
void ambc_set_walk_threads(uint64_t min_bytes, unsigned threads);
uint64_t ambc_scan_state_bytes(void);

/* pinned host memory helpers for callers without their own allocator */
void *ambc_host_alloc(uint64_t bytes);
void ambc_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* AMBC_H */
