// xz.cuh -- method id 7 (LZMACompression): decode with the semantics of Python's lzma.decompress(data) in its
// default FORMAT_AUTO, which calls liblzma's auto decoder once per stream.  What is restated here is the published
// .xz format (stream header and footer, block header, LZMA2 chunks, index, block padding, None / CRC32 / CRC64
// checks), the legacy .lzma ("alone") header, and the LZMA decoder itself (range coder, lc / lp / pb, literal, match
// and rep0..3 coding, length and distance coders), with liblzma 5.4's validity checks.  Filter chains other than a
// lone LZMA2 and the SHA-256 check are not implemented: such a stream counts as an error.
// Serial (one thread); usable from host code too, so that it can be checked against stock lzma without a device.
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>

#ifndef STD_HD
#define STD_HD __host__ __device__
#endif

struct XzCrc32Tab { uint32_t v[256]; };
struct XzCrc64Tab { uint64_t v[256]; };
constexpr XzCrc32Tab xz_make_crc32()
{
    XzCrc32Tab t{};
    for (uint32_t i = 0; i < 256; i++) {
        uint32_t c = i;
        for (int k = 0; k < 8; k++) c = (c & 1u) ? (c >> 1) ^ 0xEDB88320u : c >> 1;
        t.v[i] = c;
    }
    return t;
}
constexpr XzCrc64Tab xz_make_crc64() // ECMA-182, reflected
{
    XzCrc64Tab t{};
    for (uint64_t i = 0; i < 256; i++) {
        uint64_t c = i;
        for (int k = 0; k < 8; k++) c = (c & 1u) ? (c >> 1) ^ 0xC96C5795D7870F42ull : c >> 1;
        t.v[i] = c;
    }
    return t;
}
__constant__ XzCrc32Tab c_xz_crc32 = xz_make_crc32();
__constant__ XzCrc64Tab c_xz_crc64 = xz_make_crc64();
static constexpr XzCrc32Tab h_xz_crc32 = xz_make_crc32();
static constexpr XzCrc64Tab h_xz_crc64 = xz_make_crc64();
#ifdef __CUDA_ARCH__
#define XZ_CRC32(i) c_xz_crc32.v[i]
#define XZ_CRC64(i) c_xz_crc64.v[i]
#else
#define XZ_CRC32(i) h_xz_crc32.v[i]
#define XZ_CRC64(i) h_xz_crc64.v[i]
#endif

STD_HD inline uint32_t xz_crc32(const uint8_t *p, long n, uint32_t crc = 0)
{
    crc = ~crc;
    for (long i = 0; i < n; i++) crc = XZ_CRC32((crc ^ p[i]) & 0xFFu) ^ (crc >> 8);
    return ~crc;
}
STD_HD inline uint64_t xz_crc64(const uint8_t *p, long n)
{
    uint64_t crc = ~0ull;
    for (long i = 0; i < n; i++) crc = XZ_CRC64((crc ^ p[i]) & 0xFFu) ^ (crc >> 8);
    return ~crc;
}

// probability model: fixed part, then 0x300 << (lc + lp) literal probabilities (lc + lp <= 4)
#define LZ_IS_MATCH 0
#define LZ_IS_REP 192
#define LZ_IS_REP0 204
#define LZ_IS_REP1 216
#define LZ_IS_REP2 228
#define LZ_IS_REP0_LONG 240
#define LZ_POS_SLOT 432
#define LZ_SPEC_POS 688
#define LZ_ALIGN 802
#define LZ_LEN 818
#define LZ_REP_LEN 1332
#define LZ_LITERAL 1846
#define LZMA_PROBS_MAX (LZ_LITERAL + (0x300 << 4)) // 14134 probabilities, 28268 bytes

// outcome of one stream / step, as lzma.decompress tells them apart for the streams behind the first
#define XZ_OK 0
#define XZ_ERR 1   // liblzma reports an error (LZMAError)
#define XZ_TRUNC 2 // the input ends first (LZMAError "Compressed data ended before the end-of-stream marker ...")
#define XZ_ROOM 3  // the output would pass the buffer: decoding stops there, nothing behind it is verified

struct XzRc { // range decoder over in[pos .. lim); a read at lim sets `over`
    const uint8_t *in;
    long pos, lim;
    uint32_t range, code;
    bool over;
};
STD_HD inline void rc_norm(XzRc &rc)
{
    if (rc.range < (1u << 24)) {
        uint32_t byte = 0;
        if (rc.pos < rc.lim) byte = rc.in[rc.pos];
        else rc.over = true;
        rc.pos++;
        rc.range <<= 8;
        rc.code = (rc.code << 8) | byte;
    }
}
STD_HD inline uint32_t rc_bit(XzRc &rc, uint16_t *p)
{
    rc_norm(rc);
    const uint32_t bound = (rc.range >> 11) * *p;
    if (rc.code < bound) {
        rc.range = bound;
        *p += (2048 - *p) >> 5;
        return 0;
    }
    rc.range -= bound;
    rc.code -= bound;
    *p -= *p >> 5;
    return 1;
}
STD_HD inline uint32_t rc_tree(XzRc &rc, uint16_t *p, int nbits)
{
    uint32_t m = 1;
    for (int i = 0; i < nbits; i++) m = (m << 1) | rc_bit(rc, p + m);
    return m - (1u << nbits);
}
STD_HD inline uint32_t rc_rtree(XzRc &rc, uint16_t *p, int nbits)
{
    uint32_t m = 1, s = 0;
    for (int i = 0; i < nbits; i++) {
        const uint32_t b = rc_bit(rc, p + m);
        m = (m << 1) | b;
        s |= b << i;
    }
    return s;
}
STD_HD inline uint32_t rc_len(XzRc &rc, uint16_t *p, uint32_t ps)
{
    if (!rc_bit(rc, p)) return rc_tree(rc, p + 2 + ps * 8, 3);
    if (!rc_bit(rc, p + 1)) return 8 + rc_tree(rc, p + 130 + ps * 8, 3);
    return 16 + rc_tree(rc, p + 258, 8);
}

struct Lzma { // decoder state kept across LZMA2 chunks
    uint16_t *probs;
    uint32_t lc, lp, pb, state, rep0, rep1, rep2, rep3;
    long dict_start; // output position of the last dictionary reset
    long dsz;        // dictionary size as liblzma allocates it (>= 4096, multiple of 16)
};
STD_HD inline void lzma_reset(Lzma &z)
{
    const int n = LZ_LITERAL + (0x300 << (z.lc + z.lp));
    for (int i = 0; i < n; i++) z.probs[i] = 1024;
    z.state = 0;
    z.rep0 = z.rep1 = z.rep2 = z.rep3 = 0;
}
STD_HD inline bool lzma_props(Lzma &z, uint32_t b) // lzma_lzma_lclppb_decode; false: invalid
{
    if (b > (4 * 5 + 4) * 9 + 8) return false;
    z.pb = b / 45; b -= z.pb * 45;
    z.lp = b / 9;
    z.lc = b - z.lp * 9;
    return z.lc + z.lp <= 4;
}
STD_HD inline long lzma_dict_alloc(uint64_t d)
{
    if (d < 4096) d = 4096;
    return (long)((d + 15) & ~15ull);
}

// Decode LZMA symbols into out[*o ..) from in[pos ..) until the output reaches `stop` (a size is known: LZMA2 chunk or
// .lzma with a size) or until the end-of-payload marker (stop < 0).  allow_eopm: the marker may follow a known size.
// chunk_end: the input the symbols may use (a read behind it is an error when it exists, a truncation otherwise).
STD_HD inline int lzma_run(Lzma &z, const uint8_t *in, long len, long pos, long chunk_end, uint8_t *out, long bufsz,
                           long *o_io, long stop, bool allow_eopm, long *in_end)
{
    XzRc rc;
    rc.in = in; rc.pos = pos; rc.lim = chunk_end < len ? chunk_end : len; rc.over = false;
    const int over_kind = chunk_end <= len ? XZ_ERR : XZ_TRUNC;
    // range coder init: five bytes, the first one zero
    if (rc.pos >= rc.lim) return over_kind;
    if (in[rc.pos] != 0) return XZ_ERR;
    if (rc.pos + 5 > rc.lim) return over_kind;
    rc.code = 0;
    for (int k = 0; k < 5; k++) rc.code = (rc.code << 8) | in[rc.pos++];
    rc.range = 0xFFFFFFFFu;
    long o = *o_io;
    uint16_t *const P = z.probs;
    const uint32_t pbm = (1u << z.pb) - 1, lpm = (1u << z.lp) - 1;
#define LZ_FAIL(kind) do { *o_io = o; return rc.over ? over_kind : (kind); } while (0)
    for (;;) {
        if (rc.over) LZ_FAIL(XZ_ERR);
        if (stop >= 0 && o == stop) {
            rc_norm(rc);
            if (rc.over) LZ_FAIL(XZ_ERR);
            if (rc.code == 0) break;
            if (!allow_eopm) LZ_FAIL(XZ_ERR);
        }
        const long dpos = o - z.dict_start;
        const uint32_t ps = (uint32_t)dpos & pbm;
        const uint32_t st = z.state;
        if (!rc_bit(rc, P + LZ_IS_MATCH + st * 16 + ps)) { // literal
            if (stop >= 0 && o == stop) LZ_FAIL(XZ_ERR);
            const uint32_t prev = dpos > 0 ? out[o - 1] : 0;
            uint16_t *lp = P + LZ_LITERAL + 0x300 * ((((uint32_t)dpos & lpm) << z.lc) + (prev >> (8 - z.lc)));
            uint32_t sym = 1;
            if (st < 7) {
                while (sym < 0x100) sym = (sym << 1) | rc_bit(rc, lp + sym);
            } else {
                uint32_t mb = out[o - z.rep0 - 1], offs = 0x100;
                while (sym < 0x100) {
                    mb <<= 1;
                    const uint32_t bit = mb & offs;
                    const uint32_t b = rc_bit(rc, lp + offs + bit + sym);
                    sym = (sym << 1) | b;
                    offs &= b ? bit : ~bit;
                }
            }
            if (rc.over) LZ_FAIL(XZ_ERR);
            if (o >= bufsz) { *o_io = o; return XZ_ROOM; }
            out[o++] = (uint8_t)sym;
            z.state = st < 4 ? 0 : (st < 10 ? st - 3 : st - 6);
            continue;
        }
        uint32_t mlen;
        if (!rc_bit(rc, P + LZ_IS_REP + st)) { // match
            mlen = rc_len(rc, P + LZ_LEN, ps);
            const uint32_t ls = mlen < 4 ? mlen : 3;
            const uint32_t slot = rc_tree(rc, P + LZ_POS_SLOT + ls * 64, 6);
            uint32_t dist;
            if (slot < 4) dist = slot;
            else {
                const int nd = (int)(slot >> 1) - 1;
                dist = (2u | (slot & 1u)) << nd;
                if (slot < 14) dist += rc_rtree(rc, P + LZ_SPEC_POS + dist - slot - 1, nd);
                else {
                    uint32_t d = 0;
                    for (int k = 0; k < nd - 4; k++) {
                        rc_norm(rc);
                        rc.range >>= 1;
                        const uint32_t bit = rc.code >= rc.range;
                        if (bit) rc.code -= rc.range;
                        d = (d << 1) | bit;
                    }
                    dist += d << 4;
                    dist += rc_rtree(rc, P + LZ_ALIGN, 4);
                }
            }
            if (rc.over) LZ_FAIL(XZ_ERR);
            if (dist == 0xFFFFFFFFu) { // end-of-payload marker
                if (stop >= 0 && !(allow_eopm && o == stop)) LZ_FAIL(XZ_ERR);
                rc_norm(rc);
                if (rc.over) LZ_FAIL(XZ_ERR);
                if (rc.code != 0) LZ_FAIL(XZ_ERR);
                break;
            }
            if (stop >= 0 && o == stop) LZ_FAIL(XZ_ERR);
            const long full = dpos < z.dsz ? dpos : z.dsz;
            if ((long)dist >= full) LZ_FAIL(XZ_ERR);
            z.rep3 = z.rep2; z.rep2 = z.rep1; z.rep1 = z.rep0; z.rep0 = dist;
            z.state = st < 7 ? 7 : 10;
        } else { // repeated match
            if (stop >= 0 && o == stop) LZ_FAIL(XZ_ERR);
            if (dpos == 0) LZ_FAIL(XZ_ERR);
            if (!rc_bit(rc, P + LZ_IS_REP0 + st)) {
                if (!rc_bit(rc, P + LZ_IS_REP0_LONG + st * 16 + ps)) { // short rep: one byte at rep0
                    if (rc.over) LZ_FAIL(XZ_ERR);
                    z.state = st < 7 ? 9 : 11;
                    if (o >= bufsz) { *o_io = o; return XZ_ROOM; }
                    out[o] = out[o - z.rep0 - 1];
                    o++;
                    continue;
                }
            } else {
                uint32_t d;
                if (!rc_bit(rc, P + LZ_IS_REP1 + st)) d = z.rep1;
                else {
                    if (!rc_bit(rc, P + LZ_IS_REP2 + st)) d = z.rep2;
                    else { d = z.rep3; z.rep3 = z.rep2; }
                    z.rep2 = z.rep1;
                }
                z.rep1 = z.rep0;
                z.rep0 = d;
            }
            mlen = rc_len(rc, P + LZ_REP_LEN, ps);
            if (rc.over) LZ_FAIL(XZ_ERR);
            z.state = st < 7 ? 8 : 11;
        }
        mlen += 2;
        const long src = o - (long)z.rep0 - 1;
        for (uint32_t k = 0; k < mlen; k++) {
            if (stop >= 0 && o == stop) LZ_FAIL(XZ_ERR); // a match may not run past the known size
            if (o >= bufsz) { *o_io = o; return XZ_ROOM; }
            out[o] = out[src + k];
            o++;
        }
    }
#undef LZ_FAIL
    *o_io = o;
    *in_end = rc.pos;
    return XZ_OK;
}

// lzma_vli_decode: up to 9 bytes, no trailing zero byte
STD_HD inline int xz_vli(const uint8_t *in, long lim, long *pos, uint64_t *v, int trunc_kind)
{
    *v = 0;
    for (int i = 0; i < 9; i++) {
        if (*pos >= lim) return trunc_kind;
        const uint8_t b = in[(*pos)++];
        *v |= (uint64_t)(b & 0x7F) << (7 * i);
        if (!(b & 0x80)) return (i > 0 && b == 0) ? XZ_ERR : XZ_OK;
    }
    return XZ_ERR;
}

// one LZMA2 stream (the data of a block) at in[pos ..)
STD_HD inline int lzma2_run(Lzma &z, const uint8_t *in, long len, long pos, uint8_t *out, long bufsz, long *o_io,
                            uint32_t dict_byte, long *in_end)
{
    z.dsz = lzma_dict_alloc(dict_byte == 40 ? 0xFFFFFFFFull : (uint64_t)(2 | (dict_byte & 1)) << (dict_byte / 2 + 11));
    bool need_props = true, need_dict_reset = true;
    long o = *o_io;
    for (;;) {
        if (pos >= len) { *o_io = o; return XZ_TRUNC; }
        const uint32_t c = in[pos++];
        if (c == 0x00) break;
        if (c >= 0xE0 || c == 1) { need_props = true; need_dict_reset = true; }
        else if (need_dict_reset) { *o_io = o; return XZ_ERR; }
        if (c >= 0x80) {
            if (c < 0xC0 && need_props) { *o_io = o; return XZ_ERR; }
        } else if (c > 2) { *o_io = o; return XZ_ERR; }
        if (need_dict_reset) { need_dict_reset = false; z.dict_start = o; }
        const int nh = c >= 0xC0 ? 5 : (c >= 0x80 ? 4 : 2);
        if (pos + nh > len) { *o_io = o; return XZ_TRUNC; }
        if (c >= 0x80) {
            const long usize = (long)(((c & 0x1Fu) << 16) + ((uint32_t)in[pos] << 8) + in[pos + 1]) + 1;
            const long csize = (long)(((uint32_t)in[pos + 2] << 8) + in[pos + 3]) + 1;
            pos += 4;
            if (c >= 0xC0) {
                need_props = false;
                if (!lzma_props(z, in[pos++])) { *o_io = o; return XZ_ERR; }
                lzma_reset(z);
            } else if (c >= 0xA0) lzma_reset(z);
            long end = 0;
            const int r = lzma_run(z, in, len, pos, pos + csize, out, bufsz, &o, o + usize, false, &end);
            if (r != XZ_OK) { *o_io = o; return r; }
            if (end != pos + csize) { *o_io = o; return XZ_ERR; }
            pos = end;
        } else {
            const long csize = (long)(((uint32_t)in[pos] << 8) + in[pos + 1]) + 1;
            pos += 2;
            for (long k = 0; k < csize; k++) {
                if (pos >= len) { *o_io = o; return XZ_TRUNC; }
                if (o >= bufsz) { *o_io = o; return XZ_ROOM; }
                out[o++] = in[pos++];
            }
        }
    }
    *o_io = o;
    *in_end = pos;
    return XZ_OK;
}

__host__ __device__ constexpr int xz_check_size(int id) { return id == 0 ? 0 : 4 << ((id - 1) / 3); }

// one .xz stream at in[start ..)
STD_HD inline int xz_stream(const uint8_t *in, long len, long start, uint8_t *out, long bufsz, long o, uint16_t *probs,
                            long *o_end, long *next)
{
    long pos = start;
    const uint8_t magic[6] = {0xFD, '7', 'z', 'X', 'Z', 0x00};
    if (pos + 12 > len) {
        for (long k = 0; pos + k < len && k < 6; k++) if (in[pos + k] != magic[k]) return XZ_ERR;
        return XZ_TRUNC;
    }
    for (int k = 0; k < 6; k++) if (in[pos + k] != magic[k]) return XZ_ERR;
    const uint32_t hcrc = in[pos + 8] | (in[pos + 9] << 8) | (in[pos + 10] << 16) | ((uint32_t)in[pos + 11] << 24);
    if (xz_crc32(in + pos + 6, 2) != hcrc) return XZ_ERR;
    if (in[pos + 6] != 0 || (in[pos + 7] & 0xF0)) return XZ_ERR;
    const int check = in[pos + 7] & 0x0F;
    const uint8_t flag0 = in[pos + 6], flag1 = in[pos + 7];
    if (check == 0x0A) return XZ_ERR; // SHA-256 is not implemented
    const int csz = xz_check_size(check);
    pos += 12;
    Lzma z;
    z.probs = probs;
    uint64_t n_blocks = 0, sum_unpadded = 0, sum_uncomp = 0, hash = 0;
    for (;;) { // blocks
        if (pos >= len) return XZ_TRUNC;
        if (in[pos] == 0x00) break; // index indicator
        const long hsize = ((long)in[pos] + 1) * 4;
        if (pos + hsize > len) return XZ_TRUNC;
        const uint32_t bcrc = in[pos + hsize - 4] | (in[pos + hsize - 3] << 8) | (in[pos + hsize - 2] << 16) | ((uint32_t)in[pos + hsize - 1] << 24);
        if (xz_crc32(in + pos, hsize - 4) != bcrc) return XZ_ERR;
        const uint8_t bflags = in[pos + 1];
        if (bflags & 0x3C) return XZ_ERR;
        long hp = pos + 2;
        const long hend = pos + hsize - 4;
        uint64_t want_comp = ~0ull, want_uncomp = ~0ull;
        if (bflags & 0x40) {
            if (xz_vli(in, hend, &hp, &want_comp, XZ_ERR) != XZ_OK || want_comp == 0) return XZ_ERR;
        }
        if (bflags & 0x80) {
            if (xz_vli(in, hend, &hp, &want_uncomp, XZ_ERR) != XZ_OK) return XZ_ERR;
        }
        if ((bflags & 3) != 0) return XZ_ERR; // filter chains other than a lone LZMA2
        uint64_t fid, psize;
        if (xz_vli(in, hend, &hp, &fid, XZ_ERR) != XZ_OK || xz_vli(in, hend, &hp, &psize, XZ_ERR) != XZ_OK) return XZ_ERR;
        if (fid != 0x21 || psize != 1 || hp >= hend) return XZ_ERR;
        const uint32_t dict_byte = in[hp++];
        if ((dict_byte & 0xC0) || dict_byte > 40) return XZ_ERR;
        for (; hp < hend; hp++) if (in[hp]) return XZ_ERR; // header padding
        pos += hsize;
        const long data = pos, o0 = o;
        long end = 0;
        const int r = lzma2_run(z, in, len, pos, out, bufsz, &o, dict_byte, &end);
        if (r != XZ_OK) return r;
        const uint64_t comp = (uint64_t)(end - data), uncomp = (uint64_t)(o - o0);
        if ((want_comp != ~0ull && want_comp != comp) || (want_uncomp != ~0ull && want_uncomp != uncomp)) return XZ_ERR;
        pos = end;
        for (uint64_t k = comp; k & 3; k++) { // block padding
            if (pos >= len) return XZ_TRUNC;
            if (in[pos++]) return XZ_ERR;
        }
        if (pos + csz > len) return XZ_TRUNC;
        if (check == 1) {
            const uint32_t want = in[pos] | (in[pos + 1] << 8) | (in[pos + 2] << 16) | ((uint32_t)in[pos + 3] << 24);
            if (xz_crc32(out + o0, (long)uncomp) != want) return XZ_ERR;
        } else if (check == 4) {
            uint64_t want = 0;
            for (int k = 7; k >= 0; k--) want = (want << 8) | in[pos + k];
            if (xz_crc64(out + o0, (long)uncomp) != want) return XZ_ERR;
        }
        pos += csz;
        const uint64_t unpadded = (uint64_t)hsize + comp + (uint64_t)csz;
        n_blocks++;
        sum_unpadded += unpadded;
        sum_uncomp += uncomp;
        hash = (hash ^ unpadded) * 0x100000001B3ull;
        hash = (hash ^ uncomp) * 0x100000001B3ull;
    }
    // index
    const long index_start = pos;
    pos++;
    uint64_t count, h2 = 0;
    int r = xz_vli(in, len, &pos, &count, XZ_TRUNC);
    if (r) return r;
    if (count != n_blocks) return XZ_ERR;
    uint64_t s_unp = 0, s_unc = 0;
    for (uint64_t i = 0; i < count; i++) {
        uint64_t unp, unc;
        if ((r = xz_vli(in, len, &pos, &unp, XZ_TRUNC))) return r;
        if (unp < 5 || unp > (~0ull >> 1) - 3) return XZ_ERR;
        if ((r = xz_vli(in, len, &pos, &unc, XZ_TRUNC))) return r;
        s_unp += unp; s_unc += unc;
        h2 = (h2 ^ unp) * 0x100000001B3ull;
        h2 = (h2 ^ unc) * 0x100000001B3ull;
    }
    if (s_unp != sum_unpadded || s_unc != sum_uncomp || h2 != hash) return XZ_ERR;
    while ((pos - index_start) & 3) {
        if (pos >= len) return XZ_TRUNC;
        if (in[pos++]) return XZ_ERR;
    }
    if (pos + 4 > len) return XZ_TRUNC;
    const uint32_t icrc = in[pos] | (in[pos + 1] << 8) | (in[pos + 2] << 16) | ((uint32_t)in[pos + 3] << 24);
    if (xz_crc32(in + index_start, pos - index_start) != icrc) return XZ_ERR;
    pos += 4;
    const long index_size = pos - index_start;
    // footer
    if (pos + 12 > len) return XZ_TRUNC;
    const uint8_t *f = in + pos;
    if (f[10] != 'Y' || f[11] != 'Z') return XZ_ERR;
    const uint32_t fcrc = f[0] | (f[1] << 8) | (f[2] << 16) | ((uint32_t)f[3] << 24);
    if (xz_crc32(f + 4, 6) != fcrc) return XZ_ERR;
    const uint64_t backward = ((uint64_t)(f[4] | (f[5] << 8) | (f[6] << 16) | ((uint32_t)f[7] << 24)) + 1) * 4;
    if (f[8] != flag0 || f[9] != flag1 || backward != (uint64_t)index_size) return XZ_ERR;
    *o_end = o;
    *next = pos + 12;
    return XZ_OK;
}

// one .lzma ("alone") stream at in[start ..): 13-byte header, then LZMA1 (liblzma's picky header checks, as the auto
// decoder uses them)
STD_HD inline int alone_stream(const uint8_t *in, long len, long start, uint8_t *out, long bufsz, long o,
                               uint16_t *probs, long *o_end, long *next)
{
    long pos = start;
    Lzma z;
    z.probs = probs;
    if (pos >= len) return XZ_TRUNC;
    if (!lzma_props(z, in[pos])) return XZ_ERR;
    if (pos + 5 > len) return XZ_TRUNC;
    const uint32_t d = in[pos + 1] | (in[pos + 2] << 8) | (in[pos + 3] << 16) | ((uint32_t)in[pos + 4] << 24);
    if (d != 0xFFFFFFFFu) { // 2^n or 2^n + 2^(n-1)
        uint32_t m = d - 1;
        m |= m >> 2; m |= m >> 3; m |= m >> 4; m |= m >> 8; m |= m >> 16;
        if (m + 1 != d) return XZ_ERR;
    }
    if (pos + 13 > len) return XZ_TRUNC;
    uint64_t usize = 0;
    for (int k = 7; k >= 0; k--) usize = (usize << 8) | in[pos + 5 + k];
    if (usize != ~0ull && usize >= (1ull << 38)) return XZ_ERR;
    pos += 13;
    z.dsz = lzma_dict_alloc(d);
    z.dict_start = o;
    lzma_reset(z);
    long end = 0;
    const long stop = usize == ~0ull ? -1 : o + (long)usize;
    const int r = lzma_run(z, in, len, pos, len + 1, out, bufsz, &o, stop, true, &end);
    if (r != XZ_OK) return r;
    *o_end = o;
    *next = end;
    return XZ_OK;
}

// lzma.decompress(in[0 .. len)) with FORMAT_AUTO.  Returns the total number of decompressed bytes (out[0 .. total)),
// -1 where lzma.decompress raises, or -2 when the output would pass bufsz (out[0 .. bufsz) holds its first bytes
// as far as they decode; nothing behind them, and no check of the block they are in, is verified).
STD_HD inline long xz_decompress(const uint8_t *in, long len, uint8_t *out, long bufsz, uint16_t *probs)
{
    long o = 0, pos = 0;
    bool first = true;
    while (pos < len) {
        long o_end = 0, next = 0;
        const int r = in[pos] == 0xFD ? xz_stream(in, len, pos, out, bufsz, o, probs, &o_end, &next)
                                      : alone_stream(in, len, pos, out, bufsz, o, probs, &o_end, &next);
        if (r == XZ_ROOM) return -2;
        if (r == XZ_TRUNC || (r == XZ_ERR && first)) return -1;
        if (r == XZ_ERR) break;
        o = o_end;
        pos = next;
        first = false;
    }
    return o;
}
