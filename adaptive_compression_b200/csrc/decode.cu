// decode.cu -- package index walk (host) and the per-package decode kernel.
// Replaces AdaptiveCompressor._adaptive_decompress (adaptive_compressor.py:396-454).
#include "ambc_internal.h"
#include "decode_codec.cuh"
#include "decode_warp.cuh"
#include "deflate.cuh"
#include <thread>
#include <cstdlib>
#include <vector>

#define RAW_PIECE 65536u

// Dictionary packages decoded one warp per package by k_decode_lz (see below)
__device__ __forceinline__ bool dlz_eligible(const ambc_pkg &e)
{
    return e.type == 2 && e.comp_len <= DLZ_MAX_COMP && e.orig_len <= 8192;
}


// nominal number of bytes the reference appends for a package, knowable without decoding
static inline uint64_t nominal_out(uint32_t type, bool known, uint32_t comp, uint32_t orig)
{
    if (!known) return comp;                       // copied through (:432-435)
    switch (type) {
    case 255: return orig;                         // pad / truncate (compression_methods.py:703-713)
    case 4: return comp == 0 ? 0 : (comp < orig ? comp : orig); // :621-638
    default: return comp == 0 ? 0 : orig;          // `if not data: return b''`
    }
}

// ---- speculative helpers of the host walk ---------------------------------------------------------
// The chain is serial (pos += header + comp_len) and every step is a cache miss in a large body.
// For bodies over 32 MiB, helper threads walk disjoint segments ahead of time: each looks for the
// first plausible package header at or after its segment start and follows the chain from there,
// recording (position, type, orig, comp).  A helper may start on a false marker, but as soon as the
// real walk lands on a recorded position the two chains coincide from there on (the successor of a
// position is a function of the bytes), so the real walk consumes the records instead of touching
// the body.  Anything a helper cannot vouch for (marker mismatch, END, truncation) simply ends its
// list; the real walk reaches that position itself and applies the reference's rule.
struct WalkRec { uint64_t pos; uint32_t type, orig, comp; };
static uint64_t g_walk_min_bytes = 32ull << 20; // bodies below this are walked by one thread
static unsigned g_walk_threads = 0;             // 0 = hardware concurrency (at most 8)
// test knob (not part of include/ambc.h): lets small bodies exercise the helper threads
extern "C" void ambc_set_walk_threads(uint64_t min_bytes, unsigned threads) { g_walk_min_bytes = min_bytes; g_walk_threads = threads; }

static void spec_walk(const uint8_t *body, uint64_t len, const uint8_t *marker, uint32_t mb, uint64_t start, uint64_t stop,
                      std::vector<WalkRec> *out)
{
    const uint64_t hdr = mb + 14;
    uint64_t scan = start;
    for (;;) {
        // first plausible header: marker, a known-looking type, k == 0, used == orig, payload inside the body
        uint64_t pos = scan;
        for (; pos + hdr <= len && pos < stop; pos++) {
            if (body[pos] != marker[0] || memcmp(body + pos, marker, mb) != 0) continue;
            const uint8_t t = body[pos + mb];
            uint32_t used, orig, comp;
            memcpy(&used, body + pos + mb + 2, 4);
            memcpy(&orig, body + pos + mb + 6, 4);
            memcpy(&comp, body + pos + mb + 10, 4);
            if ((t >= 1 && t <= 11) || t == 255)
                if (body[pos + mb + 1] == 0 && used == orig && orig != 0 && pos + hdr + comp <= len) break;
        }
        if (pos + hdr > len || pos >= stop) return;
        const uint64_t first = pos;
        const size_t mark = out->size();
        bool mismatch = false;
        while (pos < stop && pos + hdr <= len) {
            if (memcmp(body + pos, marker, mb) != 0) { mismatch = true; break; }
            WalkRec r;
            r.pos = pos;
            r.type = body[pos + mb];
            memcpy(&r.orig, body + pos + mb + 6, 4);
            memcpy(&r.comp, body + pos + mb + 10, 4);
            if (r.type == 0 || pos + hdr + r.comp > len) break;
            out->push_back(r);
            pos += hdr + r.comp;
        }
        // a chain that dies on a marker mismatch after a few steps started on marker bytes inside a
        // payload: drop it and look for the next plausible header
        if (mismatch && out->size() - mark < 4) { out->resize(mark); scan = first + 1; continue; }
        return;
    }
}

// the walk itself; emit(entry) returns false when the caller's table is full
template <class Emit>
static int index_walk(const uint8_t *body, uint64_t body_len, const uint8_t *marker, uint32_t mb, uint64_t orig_size,
                      uint32_t known_mask, Emit emit, uint64_t *n_entries, uint64_t *out_bytes)
{
    if (!marker || mb < 1 || mb > 4 || (body_len && !body)) return ambc_fail(AMBC_E_ARG, "ambc_index_host: bad argument");
    uint64_t pos = 0, o = 0, ne = 0;
    const uint64_t hdr = mb + 14;

    // helper threads for large bodies
    unsigned T = 1;
    if (body_len >= g_walk_min_bytes && body_len >= 64) {
        T = g_walk_threads;
        if (!T) { // the host cores, shared with the other ranks of this node (torchrun sets LOCAL_WORLD_SIZE)
            T = std::thread::hardware_concurrency();
            const char *lws = getenv("LOCAL_WORLD_SIZE");
            const unsigned ranks = lws ? (unsigned)atoi(lws) : 1u;
            if (ranks > 1) T /= ranks;
        }
        T = T < 2 ? 1 : (T > 8 ? 8 : T);
    }
    std::vector<std::vector<WalkRec>> recs(T);
    std::vector<std::thread> helpers;
    std::vector<uint64_t> seg_start(T + 1, body_len);
    for (unsigned t = 0; t < T; t++) seg_start[t] = body_len / T * t;
    for (unsigned t = 1; t < T; t++)
        helpers.emplace_back(spec_walk, body, body_len, marker, mb, seg_start[t], seg_start[t + 1], &recs[t]);
    struct Joiner { std::vector<std::thread> &h; ~Joiner() { for (auto &x : h) if (x.joinable()) x.join(); } } joiner{helpers};
    unsigned seg = 1;          // next helper segment the walk will enter
    size_t ri = 0;             // cursor in recs[seg]
    bool seg_joined = false;

    int rc = AMBC_OK;
    bool stop = false;
    // one package with a verified header: entries, output offset, stop rule
    auto process = [&](uint64_t payload, uint32_t type, uint32_t orig, uint32_t comp) {
        bool known = type == 255 || (type < 32 && ((known_mask >> type) & 1u));
        uint64_t nominal = nominal_out(type, known, comp, orig);
        uint64_t room = orig_size > o ? orig_size - o : 0;
        uint64_t emitn = nominal < room ? nominal : room;
        if (emitn) {
            if (!known || type == 255) {
                // plain bytes (+ zero pad): pieces of at most 64 KiB
                uint64_t done = 0;
                while (done < emitn) {
                    uint64_t piece = emitn - done < RAW_PIECE ? emitn - done : RAW_PIECE;
                    uint64_t have = comp > done ? comp - done : 0; // payload bytes left for this piece
                    ambc_pkg e;
                    e.src_off = payload + done; e.dst_off = o + done;
                    e.comp_len = (uint32_t)(have < piece ? have : piece);
                    e.orig_len = (uint32_t)piece; e.type = 255; e.out_len = (uint32_t)piece;
                    if (!emit(e, ne)) { rc = ambc_fail(AMBC_E_CAPACITY, "ambc_index_host: table too small"); stop = true; return; }
                    ne++;
                    done += piece;
                }
            } else {
                ambc_pkg e;
                e.src_off = payload; e.dst_off = o; e.comp_len = comp; e.orig_len = orig; e.type = type;
                e.out_len = (uint32_t)emitn;
                if (!emit(e, ne)) { rc = ambc_fail(AMBC_E_CAPACITY, "ambc_index_host: table too small"); stop = true; return; }
                ne++;
            }
        }
        o += nominal;
        if (o >= orig_size) stop = true;                            // :444-445
    };

    while (pos < body_len && !stop) {
        // inside a helper's segment: if the walk stands on a recorded position, take the helper's chain
        while (seg < T && pos >= seg_start[seg + 1]) { seg++; ri = 0; seg_joined = false; }
        if (seg < T && pos >= seg_start[seg]) {
            if (!seg_joined) { helpers[seg - 1].join(); seg_joined = true; }
            const std::vector<WalkRec> &R = recs[seg];
            while (ri < R.size() && R[ri].pos < pos) ri++;
            if (ri < R.size() && R[ri].pos == pos) {
                while (ri < R.size() && !stop) {
                    const WalkRec &r = R[ri++];
                    process(r.pos + hdr, r.type, r.orig, r.comp);
                    pos = r.pos + hdr + r.comp;
                }
                continue;
            }
        }
        if (pos + hdr > body_len) break;                            // :400-403
        if (memcmp(body + pos, marker, mb) != 0)                    // :405-407
            return ambc_fail(AMBC_E_MARKER, "Marker mismatch in chunk header.");
        uint32_t type = body[pos + mb];
        uint32_t orig, comp;
        memcpy(&orig, body + pos + mb + 6, 4);
        memcpy(&comp, body + pos + mb + 10, 4);
        pos += hdr;
        if (type == 0) break;                                       // :422-424
        if (pos + comp > body_len) break;                           // :425-427
        process(pos, type, orig, comp);
        pos += comp;
    }
    if (rc) return rc;
    if (n_entries) *n_entries = ne;
    if (out_bytes) *out_bytes = o < orig_size ? o : orig_size;
    return AMBC_OK;
}

extern "C" int ambc_index_host(const uint8_t *body, uint64_t body_len, const uint8_t *marker, uint32_t mb,
                               uint64_t orig_size, uint32_t known_mask, ambc_pkg *table, uint64_t table_cap,
                               uint64_t *n_entries, uint64_t *out_bytes)
{
    return index_walk(body, body_len, marker, mb, orig_size, known_mask,
                      [&](const ambc_pkg &e, uint64_t i) {
                          if (!table) return true; // counting pass
                          if (i >= table_cap) return false;
                          table[i] = e;
                          return true;
                      },
                      n_entries, out_bytes);
}

// one walk, entries handed to `sink` in order (ambc_decompress_host decodes piece-wise while walking)
int ambc_index_stream(const uint8_t *body, uint64_t body_len, const uint8_t *marker, uint32_t mb, uint64_t orig_size,
                      uint32_t known_mask, void (*sink)(void *, const ambc_pkg &), void *user, uint64_t *n_entries,
                      uint64_t *out_bytes)
{
    return index_walk(body, body_len, marker, mb, orig_size, known_mask,
                      [&](const ambc_pkg &e, uint64_t) { sink(user, e); return true; }, n_entries, out_bytes);
}

// one walk into a growing vector (ambc_decompress_host)
int ambc_index_vector(const uint8_t *body, uint64_t body_len, const uint8_t *marker, uint32_t mb, uint64_t orig_size,
                      uint32_t known_mask, std::vector<ambc_pkg> &v, uint64_t *n_entries, uint64_t *out_bytes)
{
    return index_walk(body, body_len, marker, mb, orig_size, known_mask,
                      [&](const ambc_pkg &e, uint64_t i) {
                          if (i >= v.size()) v.resize(v.size() < 1024 ? 4096 : v.size() * 2);
                          v[i] = e;
                          return true;
                      },
                      n_entries, out_bytes);
}

// ---- kernel ----------------------------------------------------------------------------------
// Decode one package (block-collective).  src/dst in global memory.  Writes min(produced, cap)
// bytes to dst and returns produced (or -1 where the reference's codec raises).
__device__ int decode_package(DecCtx &d, uint32_t type, const uint8_t *__restrict__ src, uint32_t comp,
                              uint32_t orig, uint8_t *__restrict__ dst, uint32_t cap)
{
    const bool fast = comp <= (uint32_t)d.in_cap && orig <= DEC_OUT_CAP;
    if (type == 5) { // DeflateCompression.decompress (advanced_compression.py:84-97): a zlib error gives zeros, no exception
        if (comp == 0) return 0;
        volatile int *res5 = d.red;
        if (threadIdx.x == 0) {
            InfCode *codes = (InfCode *)d.X; // 2 x 608 bytes of the 12 KiB scratch
            const long got = inflate_zlib(src, (long)comp, dst, (long)cap, false, codes, codes + 1);
            res5[24] = got < 0 ? 0 : (got < (long)cap ? (int)got : (int)cap);
        }
        __syncthreads();
        const uint32_t good = (uint32_t)res5[24];
        __syncthreads();
        for (uint32_t k = good + threadIdx.x; k < cap; k += AMBC_BLOCK) dst[k] = 0;
        return (int)orig;
    }
    if (type == 255) { // bytes + zero pad, any size up to RAW_PIECE
        if ((((uintptr_t)dst) & 15) == 0) { // the usual case (pieces start at multiples of 64 KiB of an aligned output)
            const uint32_t have = comp < cap ? comp : cap;
            copy_g2g16(dst, src, have);
            for (uint32_t i = have + threadIdx.x; i < cap; i += AMBC_BLOCK) dst[i] = 0;
            return (int)orig;
        }
        uint32_t done = 0;
        while (done < cap) {
            uint32_t piece = min(cap - done, (uint32_t)DEC_OUT_CAP);
            uint32_t have = comp > done ? min(comp - done, piece) : 0;
            copy_g2s(d.out, src + done, (int)have);
            for (uint32_t i = have + threadIdx.x; i < piece; i += AMBC_BLOCK) d.out[i] = 0;
            __syncthreads();
            copy_s2g(dst + done, d.out, (int)piece);
            __syncthreads();
            done += piece;
        }
        return (int)orig;
    }
    if (fast) {
        copy_g2s(d.in, src, (int)comp);
        for (int i = (int)comp + threadIdx.x; i < (int)dec_r16(comp) + 16; i += AMBC_BLOCK) d.in[i] = 0;
        __syncthreads();
        int produced;
        switch (type) {
        case 1: produced = dec_rle(d, (int)comp, (int)orig); break;
        case 2: produced = dec_lz(d, (int)comp, (int)orig); break;
        case 3: produced = dec_huff(d, (int)comp, (int)orig); break;
        default: produced = dec_delta(d, (int)comp, (int)orig); break;
        }
        if (produced > 0) copy_s2g(dst, d.out, (int)min((uint32_t)produced, cap));
        __syncthreads();
        return produced;
    }
    // oversized package (never written by the reference's own encoder at <= 8192-byte chunks)
    volatile int *res = d.red;
    if (type == 3) {
        HuffDec h = huffdec_scratch(d.X);
        int boff; uint32_t nbits;
        int rc = comp ? huffdec_build(d, h, src, (int)min(comp, 0x7fffffffu), &boff, &nbits) : 0;
        if (comp == 0) return 0;
        if (rc < 0) return -1;
        if (threadIdx.x == 0) {
            uint32_t o = 0, limit = orig > 1 ? orig : 1;
            int node = h.root;
            for (uint32_t q = 0; q < nbits && o < limit; q++) {
                uint32_t bit = (src[boff + (q >> 3)] >> (7 - (q & 7))) & 1;
                node = bit ? h.child1[node] : h.child0[node];
                if (node < h.K) { if (o < cap) dst[o] = (uint8_t)h.lead[node]; o++; node = h.root; }
            }
            res[24] = (int)o;
        }
    } else if (threadIdx.x == 0) {
        long r;
        if (type == 1) r = slow_rle(src, comp, orig, dst, cap);
        else if (type == 2) r = lz_walk(src, comp, orig, dst, cap);
        else r = slow_delta(src, comp, orig, dst, cap);
        res[24] = (int)r;
    }
    __syncthreads();
    int r = res[24];
    __syncthreads();
    return r;
}

#ifndef KDEC_MINB
#define KDEC_MINB 6
#endif
// The packages no warp kernel takes (raw pieces, Delta, oversized or foreign packages): one CTA per package.
// Most bodies hold none, so a CTA first looks at AMBC_BLOCK table entries at once (one per thread) and then
// decodes the few that are its business, in order.
__global__ void __launch_bounds__(AMBC_BLOCK, KDEC_MINB)
k_decode(const uint8_t *__restrict__ body, const ambc_pkg *__restrict__ table, uint64_t n_entries,
         uint8_t *__restrict__ out, int in_cap, uint32_t *status)
{
    extern __shared__ uint4 smem4[];
    __shared__ uint32_t s_mask[AMBC_WARPS];
    DecCtx d;
    decctx_carve(d, (uint8_t *)smem4, in_cap);
    // entry (blockIdx.x + k * gridDim.x) is thread k's to look at, AMBC_BLOCK entries per round
    for (uint64_t k0 = 0; blockIdx.x + k0 * gridDim.x < n_entries; k0 += AMBC_BLOCK) {
        const uint64_t mine = blockIdx.x + (k0 + threadIdx.x) * (uint64_t)gridDim.x;
        bool want = false;
        if (mine < n_entries) {
            const ambc_pkg e = table[mine];
            want = !dlz_eligible(e) && !dw_eligible(e, 8192) && e.type != 6 && e.type != 7; // (6, 7: stdcodec.cu)
        }
        const uint32_t bal = __ballot_sync(FULL_MASK, want);
        if ((threadIdx.x & 31) == 0) s_mask[threadIdx.x >> 5] = bal;
        __syncthreads();
        for (int w = 0; w < AMBC_WARPS; w++) {
            uint32_t m = s_mask[w];
            while (m) {
                const int b = __ffs(m) - 1;
                m &= m - 1;
                const uint64_t i = blockIdx.x + (k0 + 32 * w + b) * (uint64_t)gridDim.x;
                const ambc_pkg e = table[i];
                uint8_t *dst = out + e.dst_off;
                int produced = decode_package(d, e.type, body + e.src_off, e.comp_len, e.orig_len, dst, e.out_len);
                // nominal length the index assumed for this package (see nominal_out)
                uint32_t nominal = e.type == 255 ? e.orig_len
                                 : e.type == 4 ? (e.comp_len == 0 ? 0 : min(e.comp_len, e.orig_len))
                                               : (e.comp_len == 0 ? 0 : e.orig_len);
                if (produced < 0) { // codec raised: orig_len zero bytes (:440-442)
                    for (uint32_t k = threadIdx.x; k < e.out_len; k += AMBC_BLOCK) dst[k] = 0;
                    if (threadIdx.x == 0 && status) atomicAdd(&status[0], 1u);
                } else if ((uint32_t)produced != nominal) {
                    // malformed stream: the reference would shift everything after it; we keep the
                    // grid and zero the gap, and report it
                    for (uint32_t k = (uint32_t)produced + threadIdx.x; k < e.out_len; k += AMBC_BLOCK) dst[k] = 0;
                    if (threadIdx.x == 0 && status) atomicAdd(&status[1], 1u);
                }
                __syncthreads();
            }
        }
        __syncthreads();
    }
}

template <int OUTCAP> // DLZ_OUT: packages of at most 4096 bytes; DLZ_OUT_BIG: 4097 .. 8192
__global__ void __launch_bounds__(DLZ_WARPS * 32)
k_decode_lz(const uint8_t *__restrict__ body, const ambc_pkg *__restrict__ table, uint64_t n_entries,
            uint8_t *__restrict__ out, uint32_t *status)
{
    extern __shared__ uint4 smem4[];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t *buf = (uint8_t *)smem4 + (size_t)w * OUTCAP;
    // entry first + k * stride is this warp's k-th; the lanes look at 32 of them at once (one round trip to the
    // table instead of one per entry: most entries belong to another decoder)
    const uint64_t first = (uint64_t)blockIdx.x * DLZ_WARPS + w, stride = (uint64_t)gridDim.x * DLZ_WARPS;
    for (uint64_t k0 = 0; first + k0 * stride < n_entries; k0 += 32) {
        const uint64_t mine = first + (k0 + lane) * stride;
        bool want = false;
        if (mine < n_entries) {
            const ambc_pkg e = table[mine];
            want = dlz_eligible(e) && (e.orig_len <= 4096) == (OUTCAP == DLZ_OUT);
        }
        uint32_t todo = __ballot_sync(FULL_MASK, want);
        while (todo) {
            const int b = __ffs(todo) - 1;
            todo &= todo - 1;
            const ambc_pkg e = table[first + (k0 + b) * stride];
            uint8_t *dst = out + e.dst_off;
            const int produced = dec_lz_warp(body + e.src_off, (int)e.comp_len, (int)e.orig_len, buf, OUTCAP);
            const uint32_t nominal = e.comp_len == 0 ? 0 : e.orig_len;
            uint32_t good = produced < 0 ? 0u : min((uint32_t)produced, e.out_len);
            // smem -> global, 16-byte stores when the destination allows
            if ((((uintptr_t)dst) & 15) == 0) {
                const uint32_t nv = good >> 4;
                for (uint32_t k = lane; k < nv; k += 32) ((uint4 *)dst)[k] = ((const uint4 *)buf)[k];
                for (uint32_t k = (nv << 4) + lane; k < good; k += 32) dst[k] = buf[k];
            } else {
                for (uint32_t k = lane; k < good; k += 32) dst[k] = buf[k];
            }
            if (produced < 0 || (uint32_t)produced != nominal) {
                for (uint32_t k = good + lane; k < e.out_len; k += 32) dst[k] = 0;
                if (lane == 0 && status) atomicAdd(&status[produced < 0 ? 0 : 1], 1u);
            }
            __syncwarp();
        }
    }
}

// zero [end of the last entry, orig_size) -- adaptive_compressor.py:447-449
__global__ void k_zero_tail(const ambc_pkg *__restrict__ table, uint64_t n_entries, uint8_t *__restrict__ out,
                            uint64_t orig_size)
{
    uint64_t covered = 0;
    if (n_entries) { const ambc_pkg e = table[n_entries - 1]; covered = e.dst_off + e.out_len; }
    for (uint64_t i = covered + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < orig_size;
         i += (uint64_t)gridDim.x * blockDim.x)
        out[i] = 0;
}

int ambc_stdcodec_decode_table(const void *body_dev, const ambc_pkg *table_dev, uint64_t n_entries, void *out_dev,
                               uint32_t *status_dev, uint32_t known_mask, cudaStream_t stream);

// launch the decoders for table[0 .. n_entries) (no tail zeroing).  Packages of types 6 and 7 are decoded when
// their bits are set in known_mask; without them the launches are exactly those of a table of native packages.
int ambc_decode_launch(const void *body_dev, const ambc_pkg *table_dev, uint64_t n_entries, void *out_dev,
                       uint32_t *status_dev, cudaStream_t stream, uint32_t known_mask)
{
    if (n_entries == 0) return AMBC_OK;
    const int in_cap = DEC_OUT_CAP; // payloads the reference's encoder emits are < orig_len <= 8192
    size_t smem = decctx_smem_bytes(in_cap);
    static bool attr_done_dev[16] = {}; // (function attributes are per device)
    size_t lsmem = (size_t)DLZ_WARPS * DLZ_OUT, lsmem_big = (size_t)DLZ_WARPS * DLZ_OUT_BIG;
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 16) return ambc_fail(AMBC_E_ARG, "device index out of range");
    bool &attr_done = attr_done_dev[dev];
    if (!attr_done) {
        CUDA_TRY(cudaFuncSetAttribute(k_decode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(k_decode_lz<DLZ_OUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsmem));
        CUDA_TRY(cudaFuncSetAttribute(k_decode_lz<DLZ_OUT_BIG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsmem_big));
        attr_done = true;
    }
    // the two decoders touch disjoint packages: k_decode_lz runs on a side stream, forked from and
    // joined back into the caller's stream
    static cudaStream_t side[16] = {};
    static cudaEvent_t ev_fork[16] = {}, ev_join[16] = {};
    if (!side[dev]) {
        CUDA_TRY(cudaStreamCreateWithFlags(&side[dev], cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&ev_fork[dev], cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&ev_join[dev], cudaEventDisableTiming));
    }
    CUDA_TRY(cudaEventRecord(ev_fork[dev], stream));
    CUDA_TRY(cudaStreamWaitEvent(side[dev], ev_fork[dev], 0));
    unsigned lgrid = (unsigned)min<uint64_t>((n_entries + DLZ_WARPS - 1) / DLZ_WARPS, 148ull * 24);
    k_decode_lz<DLZ_OUT><<<lgrid, DLZ_WARPS * 32, lsmem, side[dev]>>>((const uint8_t *)body_dev, table_dev, n_entries,
                                                                     (uint8_t *)out_dev, status_dev);
    k_decode_lz<DLZ_OUT_BIG><<<lgrid, DLZ_WARPS * 32, lsmem_big, side[dev]>>>((const uint8_t *)body_dev, table_dev, n_entries,
                                                                             (uint8_t *)out_dev, status_dev);
    ambc_count_launch();
    ambc_count_launch();
    CUDA_TRY(cudaEventRecord(ev_join[dev], side[dev]));
    // Huffman and RLE packages: 64 lanes each
    const unsigned wgrid = (unsigned)min<uint64_t>(n_entries, 148ull * 16 * 8);
    k_decode_warp<4096><<<wgrid, DW_T, DwCfg<4096>::PER_PKG, stream>>>(
        (const uint8_t *)body_dev, table_dev, n_entries, (uint8_t *)out_dev, status_dev);
    k_decode_warp<8192><<<wgrid, DW_T, DwCfg<8192>::PER_PKG, stream>>>(
        (const uint8_t *)body_dev, table_dev, n_entries, (uint8_t *)out_dev, status_dev);
    ambc_count_launch();
    ambc_count_launch();
    // everything else: one CTA each
    unsigned grid = (unsigned)min<uint64_t>(n_entries, 148ull * KDEC_MINB);
    k_decode<<<grid, AMBC_BLOCK, smem, stream>>>((const uint8_t *)body_dev, table_dev, n_entries, (uint8_t *)out_dev,
                                                 in_cap, status_dev);
    ambc_count_launch();
    if (known_mask & (AMBC_METHOD_BIT(AMBC_BZIP2) | AMBC_METHOD_BIT(AMBC_LZMA))) {
        const int rc = ambc_stdcodec_decode_table(body_dev, table_dev, n_entries, out_dev, status_dev, known_mask, stream);
        if (rc) return rc;
    }
    CUDA_TRY(cudaStreamWaitEvent(stream, ev_join[dev], 0));
    CUDA_TRY(cudaGetLastError());
    return AMBC_OK;
}

extern "C" int ambc_decompress_dev_mask(const void *body_dev, uint64_t body_len, const ambc_pkg *table_dev,
                                        uint64_t n_entries, void *out_dev, uint64_t orig_size, uint32_t known_mask,
                                        uint32_t *status_dev, void *stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    (void)body_len;
    if (orig_size && !out_dev) return ambc_fail(AMBC_E_ARG, "ambc_decompress_dev: null output");
    if (n_entries == 0) {
        if (orig_size) CUDA_TRY(cudaMemsetAsync(out_dev, 0, orig_size, stream));
        return AMBC_OK;
    }
    if (!body_dev || !table_dev) return ambc_fail(AMBC_E_ARG, "ambc_decompress_dev: null buffer");
    ambc_timing_mark(4, stream);
    k_zero_tail<<<148, 256, 0, stream>>>(table_dev, n_entries, (uint8_t *)out_dev, orig_size);
    ambc_count_launch();
    int rc = ambc_decode_launch(body_dev, table_dev, n_entries, out_dev, status_dev, stream, known_mask);
    if (rc) return rc;
    ambc_timing_mark(5, stream);
    ambc_timing().pending_d = ambc_timing().on;
    return AMBC_OK;
}

extern "C" int ambc_decompress_dev(const void *body_dev, uint64_t body_len, const ambc_pkg *table_dev,
                                   uint64_t n_entries, void *out_dev, uint64_t orig_size, uint32_t *status_dev,
                                   void *stream_)
{
    return ambc_decompress_dev_mask(body_dev, body_len, table_dev, n_entries, out_dev, orig_size, 0u, status_dev, stream_);
}

int ambc_inflate_batch(const void *in_dev, const uint64_t *in_off_dev, const uint32_t *orig_len_dev, uint32_t n_items,
                       void *out_dev, uint64_t out_stride, int32_t *out_len_dev, cudaStream_t stream);
int ambc_stdcodec_decode_batch(int method, const void *in_dev, const uint64_t *in_off_dev, const uint32_t *orig_len_dev,
                               uint32_t n_items, void *out_dev, uint64_t out_stride, int32_t *out_len_dev, cudaStream_t stream);

// ---- codec plug-in batch kernels (CompressionMethod API parity) -------------------------------
// items the warp decoders take (the same code as the container path, so the codec-level fixtures hold it too)
__device__ __forceinline__ bool codec_item_warp(int method, uint32_t comp, uint32_t orig)
{
    return (method == 1 || method == 3) && comp <= 8192u && orig <= 8192u;
}

__global__ void __launch_bounds__(DW_T)
k_codec_decode_warp(int method, const uint8_t *__restrict__ in, const uint64_t *__restrict__ in_off,
                    const uint32_t *__restrict__ orig_len, uint32_t n_items, uint8_t *__restrict__ out,
                    uint64_t out_stride, int32_t *__restrict__ out_len)
{
    extern __shared__ uint4 smem4[];
    DwCtx d;
    dw_carve<8192>(d, (uint8_t *)smem4);
    for (uint32_t i = blockIdx.x; i < n_items; i += gridDim.x) {
        const uint64_t a = in_off[i], b = in_off[i + 1];
        const uint32_t comp = (uint32_t)(b - a), orig = orig_len[i];
        if (b - a > 8192u || !codec_item_warp(method, comp, orig)) continue;
        const uint32_t cap = out_stride > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)out_stride;
        const int produced = method == 3 ? dw_huff<8192>(d, in + a, (int)comp, (int)orig) : dw_rle<8192>(d, in + a, (int)comp, (int)orig);
        if (produced > 0) dw_store(out + (uint64_t)i * out_stride, d.out, min((uint32_t)produced, cap));
        if (threadIdx.x == 0) out_len[i] = produced;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(AMBC_BLOCK)
k_codec_decode(int method, const uint8_t *__restrict__ in, const uint64_t *__restrict__ in_off,
               const uint32_t *__restrict__ orig_len, uint32_t n_items, uint8_t *__restrict__ out,
               uint64_t out_stride, int32_t *__restrict__ out_len, int in_cap)
{
    extern __shared__ uint4 smem4[];
    DecCtx d;
    decctx_carve(d, (uint8_t *)smem4, in_cap);
    for (uint32_t i = blockIdx.x; i < n_items; i += gridDim.x) {
        uint64_t a = in_off[i], b = in_off[i + 1];
        uint32_t comp = (uint32_t)(b - a), orig = orig_len[i];
        if (b - a <= 8192u && codec_item_warp(method, comp, orig)) continue; // k_codec_decode_warp
        uint32_t cap = out_stride > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)out_stride;
        int produced;
        if (method == 255) {
            // NoCompression.decompress: pad / truncate to orig (compression_methods.py:691-713)
            uint32_t done = 0, want = min(orig, cap);
            while (done < want) {
                uint32_t piece = min(want - done, (uint32_t)RAW_PIECE);
                decode_package(d, 255, in + a + done, comp > done ? comp - done : 0, piece, out + (uint64_t)i * out_stride + done, piece);
                done += piece;
            }
            produced = (int)orig;
        } else {
            produced = decode_package(d, (uint32_t)method, in + a, comp, orig, out + (uint64_t)i * out_stride, cap);
        }
        if (threadIdx.x == 0) out_len[i] = produced;
        __syncthreads();
    }
}

extern "C" int ambc_codec_decode_batch(int method, const void *in_dev, const uint64_t *in_off_dev,
                                       const uint32_t *orig_len_dev, uint32_t n_items, void *out_dev,
                                       uint64_t out_stride, int32_t *out_len_dev, void *stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!((method >= 1 && method <= 7) || method == 255))
        return ambc_fail(AMBC_E_ARG, "ambc_codec_decode_batch: unknown method %d", method);
    if (n_items == 0) return AMBC_OK;
    if (!in_off_dev || !orig_len_dev || !out_dev || !out_len_dev) return ambc_fail(AMBC_E_ARG, "null buffer");
    if (method == 5) return ambc_inflate_batch(in_dev, in_off_dev, orig_len_dev, n_items, out_dev, out_stride, out_len_dev, stream);
    if (method == 6 || method == 7)
        return ambc_stdcodec_decode_batch(method, in_dev, in_off_dev, orig_len_dev, n_items, out_dev, out_stride, out_len_dev, stream);
    const int in_cap = 2 * AMBC_NMAX + 2048; // any payload the encoders can emit for <= 8192 bytes
    size_t smem = decctx_smem_bytes(in_cap);
    CUDA_TRY(cudaFuncSetAttribute(k_codec_decode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (method == 1 || method == 3) {
        k_codec_decode_warp<<<n_items, DW_T, DwCfg<8192>::PER_PKG, stream>>>(
            method, (const uint8_t *)in_dev, in_off_dev, orig_len_dev, n_items, (uint8_t *)out_dev, out_stride, out_len_dev);
        ambc_count_launch();
    }
    k_codec_decode<<<n_items, AMBC_BLOCK, smem, stream>>>(method, (const uint8_t *)in_dev, in_off_dev, orig_len_dev,
                                                          n_items, (uint8_t *)out_dev, out_stride, out_len_dev, in_cap);
    ambc_count_launch();
    CUDA_TRY(cudaGetLastError());
    return AMBC_OK;
}
