// bzip2.cuh -- method id 6 (BZip2Compression): decode with the semantics of Python's bz2.decompress(data), which
// calls libbzip2 once per stream.  What is restated here is the published bzip2 format (stream header "BZh1".."BZh9",
// blocks with 2..6 Huffman tables, MTF-coded selectors, delta-coded code lengths, RUNA / RUNB zero runs, inverse MTF,
// inverse BWT from origPtr, the run-of-4 length bytes, randomised blocks, block CRC and combined stream CRC) with
// libbzip2 1.0.8's validity checks, so that a stream is refused exactly where the stock library refuses it.
// Serial (one thread); usable from host code too, so that it can be checked against stock bz2 without a device.
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>

#ifndef STD_HD
#define STD_HD __host__ __device__
#endif

#define BZ2_MAX_GROUPS 6
#define BZ2_MAX_ALPHA 258
#define BZ2_MAX_CODE_LEN 23
#define BZ2_MAX_SELECTORS 18002
#define BZ2_MAX_BLOCK 900000 // 100000 * the largest block-size digit: entries of the tt scratch a stream may need

struct Bz2CrcTab { uint32_t v[256]; };
constexpr Bz2CrcTab bz2_make_crc() // CRC-32, MSB first, polynomial 0x04C11DB7 (libbzip2's BZ2_crc32Table)
{
    Bz2CrcTab t{};
    for (uint32_t i = 0; i < 256; i++) {
        uint32_t c = i << 24;
        for (int k = 0; k < 8; k++) c = (c & 0x80000000u) ? (c << 1) ^ 0x04C11DB7u : c << 1;
        t.v[i] = c;
    }
    return t;
}
__constant__ Bz2CrcTab c_bz2_crc = bz2_make_crc();
static constexpr Bz2CrcTab h_bz2_crc = bz2_make_crc();

// the pseudo-random table of randomised blocks (libbzip2's BZ2_rNums)
#define BZ2_RNUMS_INIT {                                                                                              \
    619, 720, 127, 481, 931, 816, 813, 233, 566, 247, 985, 724, 205, 454, 863, 491, 741, 242, 949, 214, 733, 859, 335, 708, 621, 574, 73, 654, 730, 472, 419, 436, \
    278, 496, 867, 210, 399, 680, 480, 51, 878, 465, 811, 169, 869, 675, 611, 697, 867, 561, 862, 687, 507, 283, 482, 129, 807, 591, 733, 623, 150, 238, 59, 379, \
    684, 877, 625, 169, 643, 105, 170, 607, 520, 932, 727, 476, 693, 425, 174, 647, 73, 122, 335, 530, 442, 853, 695, 249, 445, 515, 909, 545, 703, 919, 874, 474, \
    882, 500, 594, 612, 641, 801, 220, 162, 819, 984, 589, 513, 495, 799, 161, 604, 958, 533, 221, 400, 386, 867, 600, 782, 382, 596, 414, 171, 516, 375, 682, 485, \
    911, 276, 98, 553, 163, 354, 666, 933, 424, 341, 533, 870, 227, 730, 475, 186, 263, 647, 537, 686, 600, 224, 469, 68, 770, 919, 190, 373, 294, 822, 808, 206, \
    184, 943, 795, 384, 383, 461, 404, 758, 839, 887, 715, 67, 618, 276, 204, 918, 873, 777, 604, 560, 951, 160, 578, 722, 79, 804, 96, 409, 713, 940, 652, 934, \
    970, 447, 318, 353, 859, 672, 112, 785, 645, 863, 803, 350, 139, 93, 354, 99, 820, 908, 609, 772, 154, 274, 580, 184, 79, 626, 630, 742, 653, 282, 762, 623, \
    680, 81, 927, 626, 789, 125, 411, 521, 938, 300, 821, 78, 343, 175, 128, 250, 170, 774, 972, 275, 999, 639, 495, 78, 352, 126, 857, 956, 358, 619, 580, 124, \
    737, 594, 701, 612, 669, 112, 134, 694, 363, 992, 809, 743, 168, 974, 944, 375, 748, 52, 600, 747, 642, 182, 862, 81, 344, 805, 988, 739, 511, 655, 814, 334, \
    249, 515, 897, 955, 664, 981, 649, 113, 974, 459, 893, 228, 433, 837, 553, 268, 926, 240, 102, 654, 459, 51, 686, 754, 806, 760, 493, 403, 415, 394, 687, 700, \
    946, 670, 656, 610, 738, 392, 760, 799, 887, 653, 978, 321, 576, 617, 626, 502, 894, 679, 243, 440, 680, 879, 194, 572, 640, 724, 926, 56, 204, 700, 707, 151, \
    457, 449, 797, 195, 791, 558, 945, 679, 297, 59, 87, 824, 713, 663, 412, 693, 342, 606, 134, 108, 571, 364, 631, 212, 174, 643, 304, 329, 343, 97, 430, 751, \
    497, 314, 983, 374, 822, 928, 140, 206, 73, 263, 980, 736, 876, 478, 430, 305, 170, 514, 364, 692, 829, 82, 855, 953, 676, 246, 369, 970, 294, 750, 807, 827, \
    150, 790, 288, 923, 804, 378, 215, 828, 592, 281, 565, 555, 710, 82, 896, 831, 547, 261, 524, 462, 293, 465, 502, 56, 661, 821, 976, 991, 658, 869, 905, 758, \
    745, 193, 768, 550, 608, 933, 378, 286, 215, 979, 792, 961, 61, 688, 793, 644, 986, 403, 106, 366, 905, 644, 372, 567, 466, 434, 645, 210, 389, 550, 919, 135, \
    780, 773, 635, 389, 707, 100, 626, 958, 165, 504, 920, 176, 193, 713, 857, 265, 203, 50, 668, 108, 645, 990, 626, 197, 510, 357, 358, 850, 858, 364, 936, 638}
__constant__ uint16_t c_bz2_rnums[512] = BZ2_RNUMS_INIT;
static constexpr uint16_t h_bz2_rnums[512] = BZ2_RNUMS_INIT;

#ifdef __CUDA_ARCH__
#define BZ2_CRC(i) c_bz2_crc.v[i]
#define BZ2_RNUM(i) c_bz2_rnums[i]
#else
#define BZ2_CRC(i) h_bz2_crc.v[i]
#define BZ2_RNUM(i) h_bz2_rnums[i]
#endif

// per-decoder tables (about 29 KiB: shared memory on the device)
struct Bz2Work {
    int32_t limit[BZ2_MAX_GROUPS][BZ2_MAX_CODE_LEN], base[BZ2_MAX_GROUPS][BZ2_MAX_CODE_LEN];
    int32_t perm[BZ2_MAX_GROUPS][BZ2_MAX_ALPHA];
    int32_t unzftab[256], cftab[257];
    int32_t minlen[BZ2_MAX_GROUPS];
    uint8_t len[BZ2_MAX_GROUPS][BZ2_MAX_ALPHA];
    uint8_t selector[BZ2_MAX_SELECTORS];
    uint8_t seq2unseq[256], mtf[256];
};

// outcome of one stream, as bz2.decompress tells them apart for the streams behind the first
#define BZ2_OK 0
#define BZ2_ERR 1   // libbzip2 reports a data error (OSError)
#define BZ2_TRUNC 2 // the input ends before the end-of-stream marker (ValueError)

struct Bz2Bits {
    const uint8_t *p;
    long len, pos;
    uint64_t buf;
    int cnt;
    bool eof;
};
STD_HD inline uint32_t bz2_bits(Bz2Bits &b, int n) // n <= 32, MSB first
{
    while (b.cnt < n) {
        if (b.pos >= b.len) { b.eof = true; return 0; }
        b.buf = (b.buf << 8) | b.p[b.pos++];
        b.cnt += 8;
    }
    b.cnt -= n;
    return (uint32_t)(b.buf >> b.cnt) & (uint32_t)((1ull << n) - 1ull);
}

// BZ2_hbCreateDecodeTables
STD_HD inline void bz2_tables(int32_t *limit, int32_t *base, int32_t *perm, const uint8_t *length, int minl, int maxl, int alpha)
{
    int pp = 0;
    for (int i = minl; i <= maxl; i++)
        for (int j = 0; j < alpha; j++)
            if (length[j] == i) perm[pp++] = j;
    for (int i = 0; i < BZ2_MAX_CODE_LEN; i++) base[i] = 0;
    for (int i = 0; i < alpha; i++) base[length[i] + 1]++;
    for (int i = 1; i < BZ2_MAX_CODE_LEN; i++) base[i] += base[i - 1];
    for (int i = 0; i < BZ2_MAX_CODE_LEN; i++) limit[i] = 0;
    int vec = 0;
    for (int i = minl; i <= maxl; i++) {
        vec += base[i + 1] - base[i];
        limit[i] = vec - 1;
        vec <<= 1;
    }
    for (int i = minl + 1; i <= maxl; i++) base[i] = ((limit[i - 1] + 1) << 1) - base[i];
}

// One stream at in[start ..).  Output bytes go to out[o ..) while below cap (the rest is decoded and CRC-checked but
// not stored).  On BZ2_OK, *o_end = output position behind the stream and *next = first input byte behind it.
// tt: BZ2_MAX_BLOCK words of scratch.
STD_HD inline int bz2_stream(const uint8_t *in, long len, long start, uint8_t *out, long cap, long o, Bz2Work *w,
                             uint32_t *tt, long *o_end, long *next)
{
#define BZ_NEED(n, v) do { v = bz2_bits(b, n); if (b.eof) return BZ2_TRUNC; } while (0)
    Bz2Bits b;
    b.p = in; b.len = len; b.pos = start; b.buf = 0; b.cnt = 0; b.eof = false;
    const uint8_t hdr[3] = {'B', 'Z', 'h'};
    uint32_t v;
    for (int k = 0; k < 3; k++) { BZ_NEED(8, v); if (v != hdr[k]) return BZ2_ERR; }
    BZ_NEED(8, v);
    if (v < '1' || v > '9') return BZ2_ERR;
    const int level = (int)(v - '0');
    const int nblock_max = 100000 * level;
    for (int g = 0; g < BZ2_MAX_GROUPS; g++)
        for (int i = 0; i < BZ2_MAX_ALPHA; i++) w->perm[g][i] = 0;
    uint32_t combined = 0;
    for (;;) {
        const uint8_t blk[6] = {0x31, 0x41, 0x59, 0x26, 0x53, 0x59}, eos[6] = {0x17, 0x72, 0x45, 0x38, 0x50, 0x90};
        BZ_NEED(8, v);
        const uint8_t *magic;
        if (v == 0x17) magic = eos;
        else if (v == 0x31) magic = blk;
        else return BZ2_ERR;
        for (int k = 1; k < 6; k++) { uint32_t u; BZ_NEED(8, u); if (u != magic[k]) return BZ2_ERR; }
        uint32_t stored;
        BZ_NEED(32, stored);
        if (magic == eos) {
            if (stored != combined) return BZ2_ERR;
            *o_end = o;
            *next = b.pos;
            return BZ2_OK;
        }
        uint32_t rnd, orig_ptr;
        BZ_NEED(1, rnd);
        BZ_NEED(24, orig_ptr);
        if ((long)orig_ptr > 10 + (long)nblock_max) return BZ2_ERR;
        // symbol map
        uint32_t used16;
        BZ_NEED(16, used16);
        int n_inuse = 0;
        for (int i = 0; i < 16; i++)
            if (used16 & (0x8000u >> i)) {
                uint32_t u;
                BZ_NEED(16, u);
                for (int j = 0; j < 16; j++)
                    if (u & (0x8000u >> j)) w->seq2unseq[n_inuse++] = (uint8_t)(i * 16 + j);
            }
        if (n_inuse == 0) return BZ2_ERR;
        const int alpha = n_inuse + 2;
        uint32_t n_groups, n_sel;
        BZ_NEED(3, n_groups);
        if (n_groups < 2 || n_groups > BZ2_MAX_GROUPS) return BZ2_ERR;
        BZ_NEED(15, n_sel);
        if (n_sel < 1) return BZ2_ERR;
        // selectors: unary MTF indices, undone on the fly
        uint8_t pos[BZ2_MAX_GROUPS];
        for (int g = 0; g < (int)n_groups; g++) pos[g] = (uint8_t)g;
        for (uint32_t i = 0; i < n_sel; i++) {
            int j = 0;
            for (;;) {
                uint32_t u;
                BZ_NEED(1, u);
                if (!u) break;
                if (++j >= (int)n_groups) return BZ2_ERR;
            }
            if (i < BZ2_MAX_SELECTORS) {
                const uint8_t t = pos[j];
                for (; j > 0; j--) pos[j] = pos[j - 1];
                pos[0] = t;
                w->selector[i] = t;
            }
        }
        if (n_sel > BZ2_MAX_SELECTORS) n_sel = BZ2_MAX_SELECTORS;
        // code lengths, delta coded
        for (int t = 0; t < (int)n_groups; t++) {
            uint32_t curr;
            BZ_NEED(5, curr);
            for (int i = 0; i < alpha; i++) {
                for (;;) {
                    if ((int)curr < 1 || curr > 20) return BZ2_ERR;
                    uint32_t u;
                    BZ_NEED(1, u);
                    if (!u) break;
                    BZ_NEED(1, u);
                    curr = u ? curr - 1 : curr + 1;
                }
                w->len[t][i] = (uint8_t)curr;
            }
        }
        for (int t = 0; t < (int)n_groups; t++) {
            int minl = 32, maxl = 0;
            for (int i = 0; i < alpha; i++) {
                if (w->len[t][i] > maxl) maxl = w->len[t][i];
                if (w->len[t][i] < minl) minl = w->len[t][i];
            }
            bz2_tables(w->limit[t], w->base[t], w->perm[t], w->len[t], minl, maxl, alpha);
            w->minlen[t] = minl;
        }
        // Huffman symbols -> MTF / RUNA-RUNB -> the block's bytes in tt (low 8 bits)
        const int eob = n_inuse + 1;
        for (int i = 0; i < 256; i++) { w->unzftab[i] = 0; w->mtf[i] = (uint8_t)i; }
        int group_no = -1, group_pos = 0, gsel = 0;
        int nblock = 0;
        auto next_sym = [&](int *sym) -> int {
            if (group_pos == 0) {
                if (++group_no >= (int)n_sel) return BZ2_ERR;
                group_pos = 50;
                gsel = w->selector[group_no];
            }
            group_pos--;
            int zn = w->minlen[gsel];
            uint32_t zvec = bz2_bits(b, zn);
            if (b.eof) return BZ2_TRUNC;
            for (;;) {
                if (zn > 20) return BZ2_ERR;
                if ((int32_t)zvec <= w->limit[gsel][zn]) break;
                zn++;
                const uint32_t zj = bz2_bits(b, 1);
                if (b.eof) return BZ2_TRUNC;
                zvec = (zvec << 1) | zj;
            }
            const int32_t k = (int32_t)zvec - w->base[gsel][zn];
            if (k < 0 || k >= BZ2_MAX_ALPHA) return BZ2_ERR;
            *sym = w->perm[gsel][k];
            return BZ2_OK;
        };
        int sym, r;
        if ((r = next_sym(&sym))) return r;
        for (;;) {
            if (sym == eob) break;
            if (sym == 0 || sym == 1) { // RUNA / RUNB
                int es = -1, nn = 1;
                do {
                    if (nn >= 2 * 1024 * 1024) return BZ2_ERR;
                    es += (sym + 1) * nn;
                    nn <<= 1;
                    if ((r = next_sym(&sym))) return r;
                } while (sym == 0 || sym == 1);
                es++;
                const uint8_t uc = w->seq2unseq[w->mtf[0]];
                w->unzftab[uc] += es;
                for (; es > 0; es--) {
                    if (nblock >= nblock_max) return BZ2_ERR;
                    tt[nblock++] = uc;
                }
                continue;
            }
            if (nblock >= nblock_max) return BZ2_ERR;
            int nn = sym - 1; // move to front
            const uint8_t t = w->mtf[nn];
            for (; nn > 0; nn--) w->mtf[nn] = w->mtf[nn - 1];
            w->mtf[0] = t;
            const uint8_t uc = w->seq2unseq[t];
            w->unzftab[uc]++;
            tt[nblock++] = uc;
            if ((r = next_sym(&sym))) return r;
        }
        if ((int)orig_ptr >= nblock) return BZ2_ERR;
        for (int i = 0; i < 256; i++)
            if (w->unzftab[i] < 0 || w->unzftab[i] > nblock) return BZ2_ERR;
        w->cftab[0] = 0;
        for (int i = 1; i <= 256; i++) w->cftab[i] = w->cftab[i - 1] + w->unzftab[i - 1];
        // inverse BWT: the T vector
        for (int i = 0; i < nblock; i++) {
            const uint32_t uc = tt[i] & 0xFFu;
            tt[w->cftab[uc]++] |= (uint32_t)i << 8;
        }
        uint32_t tpos = tt[orig_ptr] >> 8;
        int used = 0;
        int rn_togo = 0, rt_pos = 0;
        auto get = [&](uint32_t *c) -> bool { // BZ_GET_FAST + BZ_RAND_UPD_MASK; false: corrupt
            if (tpos >= (uint32_t)nblock_max) return false;
            tpos = tt[tpos];
            uint32_t ch = tpos & 0xFFu;
            tpos >>= 8;
            if (rnd) {
                if (rn_togo == 0) { rn_togo = BZ2_RNUM(rt_pos); if (++rt_pos == 512) rt_pos = 0; }
                rn_togo--;
                ch ^= rn_togo == 1 ? 1u : 0u;
            }
            *c = ch;
            used++;
            return true;
        };
        // undo the run-of-4 coding (unRLE_obuf_to_output) and compute the block CRC
        uint32_t crc = 0xFFFFFFFFu, k0, k1;
        if (!get(&k0)) return BZ2_ERR;
        auto emit = [&](uint32_t ch, int n) {
            for (int q = 0; q < n; q++) {
                crc = (crc << 8) ^ BZ2_CRC((crc >> 24) ^ ch);
                if (o < cap) out[o] = (uint8_t)ch;
                o++;
            }
        };
        for (;;) {
            if (used == nblock + 1) break;
            if (used > nblock + 1) return BZ2_ERR;
            int run = 1;
            const uint32_t ch = k0;
            if (!get(&k1)) return BZ2_ERR;
            if (used == nblock + 1) { emit(ch, run); continue; }
            if (k1 != k0) { k0 = k1; emit(ch, run); continue; }
            run = 2;
            if (!get(&k1)) return BZ2_ERR;
            if (used == nblock + 1) { emit(ch, run); continue; }
            if (k1 != k0) { k0 = k1; emit(ch, run); continue; }
            run = 3;
            if (!get(&k1)) return BZ2_ERR;
            if (used == nblock + 1) { emit(ch, run); continue; }
            if (k1 != k0) { k0 = k1; emit(ch, run); continue; }
            if (!get(&k1)) return BZ2_ERR;
            run = (int)k1 + 4;
            if (!get(&k0)) return BZ2_ERR;
            emit(ch, run);
        }
        crc = ~crc;
        if (crc != stored) return BZ2_ERR;
        combined = ((combined << 1) | (combined >> 31)) ^ crc;
    }
#undef BZ_NEED
}

// bz2.decompress(in[0 .. len)): concatenated streams; behind the first, a stream that libbzip2 refuses ends the
// output there (trailing bytes are ignored), a truncated one makes the whole call fail.  Returns the total number
// of decompressed bytes (the first min(total, cap) are in out) or -1 where bz2.decompress raises.
STD_HD inline long bz2_decompress(const uint8_t *in, long len, uint8_t *out, long cap, Bz2Work *w, uint32_t *tt)
{
    long o = 0, pos = 0;
    bool first = true;
    while (pos < len) {
        long o_end = 0, next = 0;
        const int r = bz2_stream(in, len, pos, out, cap, o, w, tt, &o_end, &next);
        if (r == BZ2_TRUNC || (r == BZ2_ERR && first)) return -1;
        if (r == BZ2_ERR) break;
        o = o_end;
        pos = next;
        first = false;
    }
    return o;
}
