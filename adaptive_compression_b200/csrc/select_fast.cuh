// select_fast.cuh -- the chunk trial / select step (adaptive_compressor.py:537-590) for chunks of at most
// NMAX bytes: one CTA of 128 threads per chunk, ~38 KB of shared memory, five CTAs per SM.  The plug-in batch
// kernels (codec_batch.cu) run the same encoders and gates on items of any size up to NMAX.
//
// Design choices, and why:
//   * The Dictionary trial (compression_methods.py:195-234, 283-313) no longer computes the longest match of
//     all n positions.  The greedy parse visits a few hundred of them, so the match search is LAZY:
//       1. positions are bucket-sorted by a hash of their 3 bytes (stable, ascending inside a bucket): one
//          counting sort with per-warp counters (packed u16, one 64-bit word per bucket), shared atomics only;
//       2. the scatter pass also yields a bitmap "some earlier position shares my bucket" -- a superset of
//          "my 3-gram occurred before", so runs of literals are skipped with bit scans;
//       3. the parse runs as 16 speculative chains (8 lanes each, one per n/16-byte segment).  At a visited
//          position the 8 lanes compare 8 bucket entries per step against the look-ahead (ascending order:
//          the scan stops at the first entry >= p, or as soon as a candidate reaches the cap of
//          min(32, n - p) bytes); the packed key (len << 16 | 0xFFFF - pos) makes the group maximum the
//          reference's "first strictly longer match" (earliest position among the longest);
//       4. greedy chains that start at different positions meet quickly (they share every literal and the
//          end of every match shorter than the cap), so the true chain is stitched from the speculative ones:
//          a segment is re-parsed from its true entry only until it hits a position its speculative chain
//          visited.  Match results are a function of the position alone and are memoised (eval bitmap).
//     The result is exact for any input: candidates are a superset, every length is verified on the bytes.
//   * Shared-memory atomics on this part are as cheap as stores (measured: 2.6 cycles per warp instruction,
//     tools/ubench), __match_any_sync costs 64 -- it is used only for the rare lanes of a 32-position block
//     that collide in a bucket.
//   * Huffman (compression_methods.py:354-405, 472-549) is built before the Dictionary trial, so its exact
//     size is the trial's cutoff; the trial is skipped when its lower bound cannot beat it.
//   * RLE (compression_methods.py:78-114) decides from the run-boundary bitmap alone; a chunk whose RLE payload
//     is at most the smallest payload the other methods can produce skips histogram, entropy and all trials.
//
// Everything is block-collective for blockDim.x == SF_T.
#pragma once
#include "common.cuh"

#define SF_T 128                 // threads per CTA
#define SF_W (SF_T / 32)         // warps
#ifndef SF_G
#define SF_G 4                   // lanes per parse group (chain); measured: 8 -> 14.1, 4 -> 12.6, 2 -> 12.5 ms over the six corpus kinds
#endif
#define SF_NG (SF_T / SF_G)      // parse groups = speculative chains
#define SF_WSW (11 * (32 / SF_G) + 5) // words of per-warp scratch of the pooled match evaluation
#define SF_ROUND 32              // bucket entries an owner contributes per round of the pooled evaluation
#define SF_PAD 64                // zero bytes behind the chunk
static_assert(SF_W == 4, "the per-bucket counter word holds four 16-bit fields, one per warp");

// dev-only phase timeline (build with -DAMBC_PHASE_TIMING): thread 0 of every CTA adds the clock64() delta since
// its previous mark to g_sf[id]; SF_COUNT adds work counters
#ifdef AMBC_PHASE_TIMING
__device__ unsigned long long g_sf[48];
#define SF_PH_DECL long long sf_t = clock64();
#define SF_PH(id) do { if (threadIdx.x == 0) { long long now_ = clock64(); atomicAdd(&g_sf[id], (unsigned long long)(now_ - sf_t)); sf_t = now_; } } while (0)
#ifdef AMBC_PHASE_COUNT
#define SF_COUNT(id, v) atomicAdd(&g_sf[id], (unsigned long long)(v))
#else
#define SF_COUNT(id, v)
#endif
#else
#define SF_PH_DECL
#define SF_PH(id)
#define SF_COUNT(id, v)
#endif

template <int NMAX> struct SfCfg {
    static constexpr int HB = NMAX > 4096 ? 12 : 11;          // hash bits
    static constexpr int NB = 1 << HB;                        // buckets
    static constexpr int NWORDS = NMAX / 32;                  // bitmap words
    static constexpr int A_BYTES = NB * 8;                    // region A: counters | trigram set | Huffman scratch | mlen + mpos
    // region A during the parse: mm16 (packed match per position) | five bitmaps + lenhi | ... | fo16 at the end
    static_assert(A_BYTES >= NMAX * 2 + 6 * NWORDS * 4 + NB * 2, "match table + bitmaps + fo16 overlay region A");
    static constexpr int OFF_SD = 0;
    static constexpr int OFF_A = OFF_SD + NMAX + SF_PAD;
    static constexpr int OFF_ORD = OFF_A + A_BYTES;           // ord (u16 per position) | payload buffer
    static constexpr int OFF_BSTART = OFF_ORD + NMAX * 2;
    // payload capacity.  Any payload of n <= NMAX bytes fits: RLE emits at most a 2-byte pair per byte (2n), the
    // Dictionary 2 bytes per literal or 4 per match of >= 3 bytes (2n), Huffman at most 1 + 5 * 255 + 4 + n bytes
    // (K <= 255, and the reference's tree is optimal, so it is no longer than a flat 8-bit code).
    static constexpr int PAY_BYTES = 2 * NMAX;
    static_assert(PAY_BYTES == OFF_BSTART - OFF_ORD, "the payload overlays ord");
    static constexpr int OFF_BITS = OFF_BSTART + (((NB + 1) * 2 + 15) & ~15);
    static constexpr int OFF_HIST = OFF_BITS + NWORDS * 4; // (only the run-boundary bitmap lives outside region A)
    static constexpr int OFF_HCODE = OFF_HIST + 1024;
    static constexpr int OFF_MISC = OFF_HCODE + 1280;
    #ifndef SF_EXTRA_SMEM
#define SF_EXTRA_SMEM 0 // dev knob: pad the CTA's shared memory to lower the occupancy (latency-sensitivity experiments)
#endif
    static constexpr int SMEM = OFF_MISC + 128 + 16 * SF_NG + ((SF_W * SF_WSW * 4 + 15) & ~15) + SF_EXTRA_SMEM;
};

template <int NMAX> struct SfCtx {
    uint8_t *sd;         // chunk bytes + SF_PAD zero bytes
    uint8_t *A;          // region A
    uint16_t *ord;       // bucket-sorted positions
    uint8_t *pay;        // winner's payload (overlays ord)
    uint16_t *bstart;    // NB + 1 bucket starts
    uint32_t *bmask;     // run-boundary bitmap, NWORDS words
    uint32_t *has3, *eval, *vis, *vis2, *ism, *lenhi; // bitmaps of the Dictionary trial, NWORDS words each, inside region A
    uint32_t *hist;      // 256 byte counts
    uint32_t *hcode;     // [256] Huffman code by symbol
    uint8_t *hlen;       // [256] Huffman code length by symbol
    int *red;            // 32 ints of reduction scratch
    int *gst;            // group state: 4 x SF_NG ints
    uint32_t *wsc;       // per-warp scratch of the pooled match evaluation: SF_W x SF_WSW words
    uint32_t sdb, ordb, bstb; // 32-bit shared-window addresses of sd / ord / bstart (ld.shared with 32-bit address math)
    int n;
    // views of region A
    // match of an evaluated position: (distance - 1) | (length - 3) & 15 << 12, bit 4 of length - 3 in lenhi
    __device__ __forceinline__ uint16_t *mm16() const { return (uint16_t *)A; }
    __device__ __forceinline__ uint16_t *fo16() const { return (uint16_t *)(A + SfCfg<NMAX>::A_BYTES - 2 * SfCfg<NMAX>::NB); } // NB entries
    __device__ __forceinline__ int match_len(int p) const
    {
        const uint32_t bit = 1u << (p & 31);
        if (!(ism[p >> 5] & bit)) return 0;
        return 3 + (int)(mm16()[p] >> 12) + ((lenhi[p >> 5] & bit) ? 16 : 0);
    }
};

template <int NMAX> __device__ __forceinline__ void sf_carve(SfCtx<NMAX> &c, uint8_t *base)
{
    using C = SfCfg<NMAX>;
    c.sd = base + C::OFF_SD;
    c.A = base + C::OFF_A;
    c.ord = (uint16_t *)(base + C::OFF_ORD);
    c.pay = base + C::OFF_ORD;
    c.bstart = (uint16_t *)(base + C::OFF_BSTART);
    c.bmask = (uint32_t *)(base + C::OFF_BITS);
    uint32_t *b = (uint32_t *)(c.A + 2 * NMAX);
    c.has3 = b; c.eval = b + C::NWORDS; c.vis = b + 2 * C::NWORDS; c.vis2 = b + 3 * C::NWORDS;
    c.ism = b + 4 * C::NWORDS; c.lenhi = b + 5 * C::NWORDS;
    c.hist = (uint32_t *)(base + C::OFF_HIST);
    c.hcode = (uint32_t *)(base + C::OFF_HCODE);
    c.hlen = base + C::OFF_HCODE + 1024;
    c.red = (int *)(base + C::OFF_MISC);
    c.gst = c.red + 32;
    c.wsc = (uint32_t *)(c.gst + 4 * SF_NG);
    c.sdb = (uint32_t)__cvta_generic_to_shared(c.sd);
    c.ordb = (uint32_t)__cvta_generic_to_shared(c.ord);
    c.bstb = (uint32_t)__cvta_generic_to_shared(c.bstart);
    c.n = 0;
}

// loads from the shared window by 32-bit address (read-only data of the parse: the chunk, ord, bstart).  Address
// arithmetic on generic pointers made ptxas emit 64-bit adds and generic LD.E for the unaligned word loads.
__device__ __forceinline__ uint32_t sf_lds32(uint32_t a) { uint32_t v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t sf_lds16(uint32_t a) { uint32_t v; asm("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t sf_lds8(uint32_t a) { uint32_t v; asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
// unaligned 32-bit load at shared-window address a
__device__ __forceinline__ uint32_t sf_ldsu(uint32_t a)
{
    const uint32_t b = a & ~3u;
    return __funnelshift_r(sf_lds32(b), sf_lds32(b + 4), (a & 3u) * 8);
}

// ---- block helpers for SF_T threads ------------------------------------------------------------------
__device__ __forceinline__ int sf_block_sum(int v, volatile int *red)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    v = __reduce_add_sync(FULL_MASK, v);
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    return red[0] + red[1] + red[2] + red[3];
}
// two sums at once
__device__ __forceinline__ void sf_block_sum2(int &a, int &b, volatile int *red)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    a = __reduce_add_sync(FULL_MASK, a);
    b = __reduce_add_sync(FULL_MASK, b);
    __syncthreads();
    if (lane == 0) { red[w] = a; red[4 + w] = b; }
    __syncthreads();
    a = red[0] + red[1] + red[2] + red[3];
    b = red[4] + red[5] + red[6] + red[7];
}
__device__ __forceinline__ int sf_block_excl_scan(int v, volatile int *red, int *total)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int inc = warp_incl_scan(v);
    __syncthreads();
    if (lane == 31) red[w] = inc;
    __syncthreads();
    const int r0 = red[0], r1 = red[1], r2 = red[2], r3 = red[3];
    *total = r0 + r1 + r2 + r3;
    const int base = (w > 0 ? r0 : 0) + (w > 1 ? r1 : 0) + (w > 2 ? r2 : 0);
    return base + inc - v;
}

__device__ __forceinline__ uint32_t sf_hash3(uint32_t tri, int hb) { return (tri * 2654435761u) >> (32 - hb); }

// ---- load ------------------------------------------------------------------------------------------------
template <int NMAX> __device__ inline void sf_load(SfCtx<NMAX> &c, const uint8_t *__restrict__ src, int n)
{
    const int tid = threadIdx.x;
    c.n = n;
    if ((((uintptr_t)src) & 15) == 0) {
        const int nv = n >> 4;
        const uint4 *s4 = (const uint4 *)src;
        uint4 *d4 = (uint4 *)c.sd;
        for (int i = tid; i < nv; i += SF_T) d4[i] = __ldg(s4 + i);
        for (int i = (nv << 4) + tid; i < n; i += SF_T) c.sd[i] = __ldg(src + i);
    } else {
        for (int i = tid; i < n; i += SF_T) c.sd[i] = __ldg(src + i);
    }
    const int padend = ((n + 15) & ~15) + SF_PAD;
    for (int i = n + tid; i < padend; i += SF_T) c.sd[i] = 0;
    __syncthreads();
}

// ---- run-boundary bitmap, RLE gate and pair count (compression_methods.py:95-109, 165-180) ---------------
// bits 0, s, 2 s, ... of a 32-bit word, by s = 1..8
static __constant__ uint32_t sf_step_mask[9] = {0x00000000u, 0xFFFFFFFFu, 0x55555555u, 0x49249249u, 0x11111111u,
                                                0x42108421u, 0x41041041u, 0x10204081u, 0x01010101u};
// bmask bit p = (p == 0 || sd[p] != sd[p-1]).  rep = sampled positions i with sd[i] == sd[i+1].
// Returns rep (block-wide); *pairs = number of (byte, count) pairs RLE emits -- computed only when the gate holds.
template <int NMAX> __device__ inline bool sf_rle_features(SfCtx<NMAX> &c, int *pairs_out)
{
    const int n = c.n, tid = threadIdx.x;
    const int nw = (n + 31) >> 5;
    const int ss = min(1000, n);
    const int step = n < 4 ? 1 : max(1, n / ss);
    // sampled positions i = 0, step, 2 step, ...: bits 0, step, 2 step, ... of a word (sf_step_mask, step <= 8 for
    // n <= 8192), shifted to the word's first sample.  Keep this branch-free: the equivalent C++ with a branch per
    // step value (S = ~0u for step 1, 0x11111111 for step 4, a bit loop otherwise) was mis-compiled by the CUDA 12.9
    // ptxas for sm_100a -- the `step == 1` branch was taken on the predicate of the VIMNMX that forms
    // max(1, n / ss), so S was ~0u for every step: rep counted all positions, and k_select_fast<4096> opened the gate
    // on 2000..4096-byte chunks the reference rejects.
    const uint32_t Sp = sf_step_mask[step];
    int rep = 0;
    for (int wd = tid; wd < nw; wd += SF_T) {
        const uint4 a = *(const uint4 *)(c.sd + 32 * wd);
        const uint4 b = *(const uint4 *)(c.sd + 32 * wd + 16);
        const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        uint32_t prevw = wd ? ((uint32_t)c.sd[32 * wd - 1] << 24) : 0;
        uint32_t mask = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const uint32_t sh = __funnelshift_l(prevw, w[k], 8); // byte j-1 under byte j
            const uint32_t x = w[k] ^ sh;
            const uint32_t y = ((x | ((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu)) & 0x80808080u) >> 7; // 1 per non-zero byte
            mask |= ((y * 0x01020408u) >> 24 & 0xFu) << (4 * k);
            prevw = w[k];
        }
        if (wd == 0) mask |= 1u;
        const int m = min(32, n - 32 * wd);
        const uint32_t valid = m == 32 ? 0xFFFFFFFFu : ((1u << m) - 1u);
        mask &= valid;
        c.bmask[wd] = mask;
        // equal-to-next bits: e[j] = sd[32wd+j] == sd[32wd+j+1], for positions below n-1
        const uint32_t nextb = (c.sd[32 * wd + 32] != (b.w >> 24)) ? 1u : 0u;
        uint32_t eq = ~((mask >> 1) | (nextb << 31));
        const int m1 = min(32, n - 1 - 32 * wd); // positions with a successor
        eq &= m1 >= 32 ? 0xFFFFFFFFu : (m1 <= 0 ? 0u : ((1u << m1) - 1u));
        const uint32_t S = Sp << ((step - (32 * wd) % step) % step);
        rep += __popc(eq & S);
    }
    rep = sf_block_sum(rep, c.red); // (also publishes bmask)
    // gate: rep / (ss - 1) > 0.3 in fp64 == 10 * rep > 3 * (ss - 1) (operands below 1000: quotients other than
    // exactly 3/10 are >= 1e-4 away from it, and the exact one rounds to the double the literal denotes)
    const bool gate = n >= 4 && 10 * rep > 3 * (ss - 1);
    if (!gate) { *pairs_out = 0; return false; }
    int pairs = 0;
    for (int wd = tid; wd < nw; wd += SF_T) {
        const uint32_t mask = c.bmask[wd];
        if (mask) {
            pairs += __popc(mask);
            // only the last run that starts in this word can be longer than 31 bytes
            const int p = 32 * wd + 31 - __clz(mask);
            int q = n;
            for (int w2 = wd + 1; w2 < nw; w2++) {
                const uint32_t m2 = c.bmask[w2];
                if (m2) { q = 32 * w2 + __ffs(m2) - 1; break; }
            }
            const int R = q - p;
            if (R > 255) pairs += (R + 254) / 255 - 1;
        }
    }
    *pairs_out = sf_block_sum(pairs, c.red);
    return true;
}

// RLE payload -> c.pay (requires bmask).  Returns the length.
template <int NMAX> __device__ inline int sf_rle_emit(SfCtx<NMAX> &c)
{
    const int n = c.n, tid = threadIdx.x;
    const int nw = (n + 31) >> 5;
    // words per thread, contiguous, so that one scan places everything (NMAX / 32 <= 2 * SF_T)
    const int wpt = (nw + SF_T - 1) / SF_T;
    int pairs = 0;
    for (int wd = tid * wpt; wd < min(nw, (tid + 1) * wpt); wd++) {
        const uint32_t mask = c.bmask[wd];
        if (mask) {
            pairs += __popc(mask);
            const int p = 32 * wd + 31 - __clz(mask);
            int q = n;
            for (int w2 = wd + 1; w2 < nw; w2++) {
                const uint32_t m2 = c.bmask[w2];
                if (m2) { q = 32 * w2 + __ffs(m2) - 1; break; }
            }
            const int R = q - p;
            if (R > 255) pairs += (R + 254) / 255 - 1;
        }
    }
    int total;
    int off = 2 * sf_block_excl_scan(pairs, c.red, &total);
    __syncthreads(); // (pay overlays nothing RLE needs, but the scan scratch is reused below)
    for (int wd = tid * wpt; wd < min(nw, (tid + 1) * wpt); wd++) {
        uint32_t mask = c.bmask[wd];
        while (mask) {
            const int bit = __ffs(mask) - 1;
            mask &= mask - 1;
            const int p = 32 * wd + bit;
            int q;
            if (mask) q = 32 * wd + __ffs(mask) - 1;
            else {
                q = n;
                for (int w2 = wd + 1; w2 < nw; w2++) {
                    const uint32_t m2 = c.bmask[w2];
                    if (m2) { q = 32 * w2 + __ffs(m2) - 1; break; }
                }
            }
            int R = q - p;
            const uint8_t v = c.sd[p];
            while (R > 0) {
                const int cnt = R > 255 ? 255 : R;
                if (off + 2 <= SfCfg<NMAX>::PAY_BYTES) { c.pay[off] = v; c.pay[off + 1] = (uint8_t)cnt; }
                off += 2;
                R -= cnt;
            }
        }
    }
    __syncthreads();
    return 2 * total;
}

// ---- histogram, distinct byte values, entropy, distinct trigrams -------------------------------------
struct SfStats { int K; int distinct3; float H; };

template <int NMAX> __device__ inline void sf_stats(SfCtx<NMAX> &c, bool want_tri, SfStats &s)
{
    const int n = c.n, tid = threadIdx.x;
    uint32_t *tri = (uint32_t *)c.A; // 2048-slot open-addressing set (8 KB of region A)
    for (int i = tid; i < 256; i += SF_T) c.hist[i] = 0;
    if (want_tri)
        for (int i = tid; i < 2048 / 4; i += SF_T) ((uint4 *)tri)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    const int nw = (n + 31) >> 5;
    for (int wd = tid; wd < nw; wd += SF_T) {
        const uint4 a = *(const uint4 *)(c.sd + 32 * wd);
        const uint4 b = *(const uint4 *)(c.sd + 32 * wd + 16);
        const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        const int m = min(32, n - 32 * wd);
        // runs of equal bytes inside the slice are added at once (text has runs of blanks, binary of zeros)
        uint32_t cur = w[0] & 0xFFu, cnt = 0;
#pragma unroll
        for (int j = 0; j < 32; j++) {
            if (j < m) {
                const uint32_t v = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
                if (v == cur) cnt++;
                else { atomicAdd(&c.hist[cur], cnt); cur = v; cnt = 1; }
            }
        }
        atomicAdd(&c.hist[cur], cnt);
    }
    // distinct trigrams among the first min(n - 3, 1000) positions (compression_methods.py:326-343)
    int ins = 0;
    if (want_tri) {
        const int cnt3 = min(n - 3, min(1000, n));
        for (int i = tid; i < cnt3; i += SF_T) {
            const uint32_t t = lds_u32u(c.sd + i) & 0xFFFFFFu;
            const uint32_t key = t + 1;
            uint32_t h = (t * 2654435761u) >> 21;
            for (;;) {
                const uint32_t old = atomicCAS(&tri[h], 0u, key);
                if (old == 0u) { ins++; break; }
                if (old == key) break;
                h = (h + 1) & 2047;
            }
        }
    }
    __syncthreads();
    // entropy in fp32 (compression_methods.py:566-574); the caller redoes near-threshold cases in fp64
    float hsum = 0.0f;
    int k = 0;
    const float inv_n = 1.0f / (float)n;
    for (int b = tid; b < 256; b += SF_T) {
        const uint32_t cnt = c.hist[b];
        if (cnt) {
            k++;
            const float p = (float)cnt * inv_n;
            hsum -= p * __log2f(p);
        }
    }
    const int lane = tid & 31, w = tid >> 5;
    k = __reduce_add_sync(FULL_MASK, k);
    ins = __reduce_add_sync(FULL_MASK, ins);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) hsum += __shfl_xor_sync(FULL_MASK, hsum, d);
    __syncthreads();
    if (lane == 0) { c.red[w] = k; c.red[4 + w] = ins; ((float *)c.red)[8 + w] = hsum; }
    __syncthreads();
    s.K = c.red[0] + c.red[1] + c.red[2] + c.red[3];
    s.distinct3 = c.red[4] + c.red[5] + c.red[6] + c.red[7];
    const float *rf = (const float *)c.red;
    s.H = (rf[8] + rf[9]) + (rf[10] + rf[11]);
    __syncthreads();
}

// ---- Huffman ---------------------------------------------------------------------------------------
// scratch inside region A (dead before the Dictionary index is built, free again after the trial)
struct SfHuff {
    uint32_t *ck;       // [256] compacted keys (count << 8 | symbol)
    uint32_t *nodeW;    // [512] (weight << 8 | leader), sorted leaves then merged nodes
    uint16_t *parent;   // [512]
    uint8_t *nbit;      // [512]
    uint8_t *leafsym;   // [256]
    uint32_t *firstpos; // [256]
    uint8_t *order;     // [256] symbols in first-occurrence order
    uint32_t *bw;       // bit words of the stream (NMAX bytes + 16), behind the rest
};
template <int NMAX> __device__ __forceinline__ SfHuff sf_huff_scratch(SfCtx<NMAX> &c)
{
    SfHuff h;
    uint8_t *X = c.A;
    h.ck = (uint32_t *)X;
    h.nodeW = (uint32_t *)(X + 1024);
    h.parent = (uint16_t *)(X + 3072);
    h.nbit = X + 4096;
    h.leafsym = X + 4608;
    h.firstpos = (uint32_t *)(X + 4864);
    h.order = X + 5888;
    h.bw = (uint32_t *)(X + 6144);
    return h;
}
static_assert(6144 + 4096 + 16 <= SfCfg<4096>::A_BYTES && 6144 + 8192 + 16 <= SfCfg<8192>::A_BYTES, "Huffman scratch fits region A");

// first-occurrence order of the byte values (Counter insertion order, compression_methods.py:368-370 / :566)
template <int NMAX> __device__ inline void sf_first_order(SfCtx<NMAX> &c, SfHuff &h, int K)
{
    const int n = c.n, tid = threadIdx.x;
    for (int i = tid; i < 256; i += SF_T) h.firstpos[i] = 0xFFFFFFFFu;
    __syncthreads();
    volatile uint32_t *fpv = h.firstpos;
    for (int s = tid; 8 * s < n; s += SF_T) { // ascending sweep: the guards fail almost always after the first pass
        const uint2 w = *(const uint2 *)(c.sd + 8 * s);
        const int m = min(8, n - 8 * s);
        uint32_t prev = 0x100u;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const uint32_t v = ((j < 4 ? w.x : w.y) >> (8 * (j & 3))) & 0xFFu;
            if (j < m && v != prev && fpv[v] > (uint32_t)(8 * s + j)) atomicMin(&h.firstpos[v], (uint32_t)(8 * s + j));
            prev = v;
        }
    }
    __syncthreads();
    // rank of each present symbol by first position (K <= 256 keys, all distinct)
    int *cntK = c.red + 16;
    if (tid == 0) *cntK = 0;
    __syncthreads();
    for (int b = tid; b < 256; b += SF_T) {
        const uint32_t fp = h.firstpos[b];
        if (fp != 0xFFFFFFFFu) h.ck[atomicAdd(cntK, 1)] = (fp << 8) | (uint32_t)b;
    }
    __syncthreads();
    for (int j = tid; j < K; j += SF_T) {
        const uint32_t key = h.ck[j];
        int r = 0;
        for (int x = 0; x < K; x++) r += (h.ck[x] < key);
        h.order[r] = (uint8_t)(key & 0xFFu);
    }
    __syncthreads();
}

// exact Python-order entropy: e -= p * log2(p) over the Counter's insertion order, no FMA contraction
template <int NMAX> __device__ inline double sf_entropy_ordered(SfCtx<NMAX> &c, SfHuff &h, int K)
{
    volatile double *out = (volatile double *)(c.red + 20);
    if (threadIdx.x == 0) {
        double e = 0.0;
        for (int r = 0; r < K; r++) {
            const double p = __ddiv_rn((double)c.hist[h.order[r]], (double)c.n);
            e = __dsub_rn(e, __dmul_rn(p, log2(p)));
        }
        out[0] = e;
    }
    __syncthreads();
    const double e = out[0];
    __syncthreads();
    return e;
}

// The reference's tree for the counts in c.hist (2 <= K <= 256): repeatedly merge the two smallest nodes under
// (weight, leader); lo gets bit 0, hi bit 1; leader(merged) = leader(lo) (compression_methods.py:482-494).
// Leaves are sorted by (weight, symbol) and merged nodes come out in that order, so two queues suffice.
// Fills c.hlen / c.hcode, returns the total number of code bits.
template <int NMAX> __device__ inline int sf_huff_build(SfCtx<NMAX> &c, SfHuff &h, int K)
{
    const int tid = threadIdx.x;
    int *cntK = c.red + 16;
    if (tid == 0) *cntK = 0;
    for (int b = tid; b < 256; b += SF_T) { c.hlen[b] = 0; c.hcode[b] = 0; }
    __syncthreads();
    for (int b = tid; b < 256; b += SF_T) {
        const uint32_t cnt = c.hist[b];
        if (cnt) h.ck[atomicAdd(cntK, 1)] = (cnt << 8) | (uint32_t)b;
    }
    __syncthreads();
    for (int j = tid; j < K; j += SF_T) { // rank sort: keys are distinct
        const uint32_t key = h.ck[j];
        int r = 0;
        for (int x = 0; x < K; x++) r += (h.ck[x] < key);
        h.nodeW[r] = key;
        h.leafsym[r] = (uint8_t)(key & 0xFFu);
    }
    __syncthreads();
    if (tid == 0) {
        int li = 0, mi = K, t = K;
        uint32_t kl = h.nodeW[0];
        uint32_t km = 0xFFFFFFFFu;
        for (int it = 0; it < K - 1; it++) {
            int pick[2];
            uint32_t pk[2];
#pragma unroll
            for (int z = 0; z < 2; z++) {
                const bool hasL = li < K, hasM = mi < t;
                const bool takeL = (hasL && hasM) ? kl < km : hasL;
                if (takeL) {
                    pick[z] = li; pk[z] = kl;
                    li++;
                    if (li < K) kl = h.nodeW[li];
                } else {
                    pick[z] = mi; pk[z] = km;
                    mi++;
                    if (mi < t) km = h.nodeW[mi];
                }
            }
            const uint32_t nk = (((pk[0] >> 8) + (pk[1] >> 8)) << 8) | (pk[0] & 0xFFu);
            h.nodeW[t] = nk;
            h.parent[pick[0]] = (uint16_t)t; h.nbit[pick[0]] = 0;
            h.parent[pick[1]] = (uint16_t)t; h.nbit[pick[1]] = 1;
            if (mi == t) km = nk;
            t++;
        }
    }
    __syncthreads();
    const int root = 2 * K - 2;
    int bits = 0;
    for (int j = tid; j < K; j += SF_T) {
        int node = j, len = 0;
        uint32_t code = 0;
        while (node != root) {
            code |= (uint32_t)h.nbit[node] << len;
            len++;
            node = h.parent[node];
        }
        const int sym = h.leafsym[j];
        c.hlen[sym] = (uint8_t)len;
        c.hcode[sym] = code;
        bits += len * (int)c.hist[sym];
    }
    return sf_block_sum(bits, c.red);
}

// Payload (table in first-occurrence order + bit count + MSB-first bit stream, compression_methods.py:379-403)
// -> c.pay.  Requires sf_huff_build (c.hcode / c.hlen) and region A free.
template <int NMAX> __device__ inline int sf_huff_emit(SfCtx<NMAX> &c, SfHuff &h, int K, int total_bits)
{
    const int n = c.n, tid = threadIdx.x;
    sf_first_order(c, h, K);
    const int hdr = 1 + 5 * K + 4;
    const int nbytes = (total_bits + 7) >> 3;
    if (tid == 0) c.pay[0] = (uint8_t)K;
    for (int r = tid; r < K; r += SF_T) {
        const int o = 1 + 5 * r;
        if (o + 5 <= SfCfg<NMAX>::PAY_BYTES) {
            const int sym = h.order[r];
            c.pay[o] = (uint8_t)sym;
            store_u32le(c.pay + o + 1, c.hist[sym]);
        }
    }
    if (tid == 0 && hdr <= SfCfg<NMAX>::PAY_BYTES) store_u32le(c.pay + hdr - 4, (uint32_t)total_bits);
    const int nwords = (total_bits + 31) >> 5;
    const int wcap = min(nwords, NMAX / 4 + 1);
    for (int i = tid; i < wcap; i += SF_T) h.bw[i] = 0;
    // 32-byte slices, contiguous per thread
    const int nsl = (n + 31) >> 5;
    const int spt = (nsl + SF_T - 1) / SF_T;
    int mybits = 0;
    for (int s = tid * spt; s < min(nsl, (tid + 1) * spt); s++) {
        const uint4 a = *(const uint4 *)(c.sd + 32 * s);
        const uint4 b = *(const uint4 *)(c.sd + 32 * s + 16);
        const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        const int m = min(32, n - 32 * s);
#pragma unroll
        for (int j = 0; j < 32; j++)
            if (j < m) mybits += c.hlen[(w[j >> 2] >> (8 * (j & 3))) & 0xFFu];
    }
    int tot;
    const int g = sf_block_excl_scan(mybits, c.red, &tot); // (its barriers also order the zeroing of bw)
    {
        int wi = g >> 5, used = g & 31;
        uint32_t cur = 0;
        bool first = true; // the first and last words of a thread may be shared with its neighbours
        for (int s = tid * spt; s < min(nsl, (tid + 1) * spt); s++) {
            const uint4 a = *(const uint4 *)(c.sd + 32 * s);
            const uint4 b = *(const uint4 *)(c.sd + 32 * s + 16);
            const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
            const int m = min(32, n - 32 * s);
#pragma unroll
            for (int j = 0; j < 32; j++) {
                if (j < m) {
                    const int sym = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
                    const uint32_t code = c.hcode[sym];
                    const int l = c.hlen[sym];
                    const int space = 32 - used;
                    if (l < space) {
                        cur |= code << (space - l);
                        used += l;
                    } else {
                        cur |= code >> (l - space);
                        if (wi < wcap) { if (first) atomicOr(&h.bw[wi], cur); else h.bw[wi] = cur; }
                        first = false;
                        wi++;
                        used = l - space;
                        cur = used ? code << (32 - used) : 0u;
                    }
                }
            }
        }
        if (used && wi < wcap) atomicOr(&h.bw[wi], cur);
    }
    __syncthreads();
    for (int k = tid; k < nbytes; k += SF_T)
        if (hdr + k < SfCfg<NMAX>::PAY_BYTES) c.pay[hdr + k] = (uint8_t)(h.bw[k >> 2] >> (24 - 8 * (k & 3)));
    __syncthreads();
    return hdr + nbytes;
}

// ---- Dictionary: index --------------------------------------------------------------------------------
// Lower bound of the Dictionary payload for n bytes: the first token is a literal, every other token covers
// at most 32 bytes (lookahead_size) for at least 2 bytes of output.
__host__ __device__ inline int sf_lz_lower_bound(int n)
{
    if (n <= 0) return 0;
    const int r = (n - 1) % 32;
    return 2 + 4 * ((n - 1) / 32) + (2 * r < 4 ? 2 * r : 4);
}

// entry of ord: position | fingerprint of the 4th byte in the spare high bits
template <int NMAX> struct SfOrd {
    static constexpr int POSB = NMAX > 4096 ? 13 : 12;
    static constexpr uint32_t POSMASK = (1u << POSB) - 1u;
    __device__ static __forceinline__ uint32_t fp(uint32_t b)
    {
        return POSB == 12 ? ((b ^ (b >> 4)) & 0xFu) : ((b ^ (b >> 2) ^ (b >> 5)) & 0x7u);
    }
};
// bucket of the position whose four bytes are w4: the top HB - 3 bits of the trigram hash (the class), then 3 bits
// of the 4th byte.  The matches of >= 4 bytes of a position lie in its own bucket, those of exactly 3 bytes in the
// 8 buckets of its class.  (With one bucket per trigram hash, zero-padded binary records put 200+ entries in front
// of every visited position: 300 k warp instructions per chunk, ncu.)
template <int NMAX> __device__ __forceinline__ uint32_t sf_bucket(uint32_t w4, uint32_t *hprod)
{
    using C = SfCfg<NMAX>;
    const uint32_t hp = (w4 & 0xFFFFFFu) * 2654435761u;
    const uint32_t b4 = w4 >> 24;
    *hprod = hp;
    return ((hp >> (32 - (C::HB - 3))) << 3) | ((b4 ^ (b4 >> 3) ^ (b4 >> 6)) & 7u);
}

// Stable bucket sort of the positions [0, n - 2) (sf_bucket; ascending inside each bucket): c.ord, c.bstart, and
// c.has3 bit p = "an earlier position has a trigram with the same HB-bit hash" (a superset of "the trigram at p
// occurred before": everything else is a literal for sure).
template <int NMAX> __device__ inline void sf_lz_index(SfCtx<NMAX> &c)
{
    using C = SfCfg<NMAX>;
    const int n = c.n, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int P = n - 2;                          // positions with 3 bytes
    const int nblk = (P + 31) >> 5;               // 32-position blocks
    const int Rw = (nblk + SF_W - 1) / SF_W;      // blocks per warp, contiguous: warp order == position order
    uint64_t *cnt64 = (uint64_t *)c.A;            // per bucket: four u16 fields, one per warp
    uint32_t *cnt32 = (uint32_t *)c.A;
    volatile uint16_t *cnt16 = (volatile uint16_t *)c.A;
    SF_PH_DECL
    for (int i = tid; i < C::NB / 2; i += SF_T) ((uint4 *)c.A)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    const uint32_t inc = (w & 1) ? 0x10000u : 1u;
    const int fsel = w >> 1;
    // pass 1: counts (order irrelevant)
    for (int r = 0; r < Rw; r++) {
        const int p = 32 * (w * Rw + r) + lane;
        if (p < P) {
            uint32_t hp;
            const uint32_t b = sf_bucket<NMAX>(sf_ldsu(c.sdb + p), &hp);
            atomicAdd(&cnt32[2 * b + fsel], inc);
        }
    }
    __syncthreads();
    SF_PH(10);
    {   // exclusive scan over (bucket-major, warp-minor); thread owns BPT consecutive buckets
        constexpr int BPT = C::NB / SF_T;
        uint64_t x[BPT];
        uint32_t run = 0;
#pragma unroll
        for (int k = 0; k < BPT; k += 2) {
            const ulonglong2 v = *(const ulonglong2 *)(cnt64 + BPT * tid + k);
            x[k] = v.x; x[k + 1] = v.y;
        }
#pragma unroll
        for (int k = 0; k < BPT; k++) {
            const uint64_t v = x[k];
            const uint64_t incl = v + (v << 16) + (v << 32) + (v << 48); // inclusive prefix of the four fields
            x[k] = (incl - v) + (uint64_t)run * 0x0001000100010001ull;
            run += (uint32_t)(incl >> 48);
        }
        int tot;
        const uint32_t base = (uint32_t)sf_block_excl_scan((int)run, c.red, &tot);
        const uint64_t b4 = (uint64_t)base * 0x0001000100010001ull;
#pragma unroll
        for (int k = 0; k < BPT; k += 2) {
            ulonglong2 v;
            v.x = x[k] + b4; v.y = x[k + 1] + b4;
            *(ulonglong2 *)(cnt64 + BPT * tid + k) = v;
            c.bstart[BPT * tid + k] = (uint16_t)v.x;
            c.bstart[BPT * tid + k + 1] = (uint16_t)v.y;
        }
        if (tid == 0) c.bstart[C::NB] = (uint16_t)P;
    }
    __syncthreads();
    SF_PH(11);
    // pass 2: ordered scatter.  A warp walks its blocks in ascending order; inside a block the lanes that share a
    // bucket (rare) are ranked by lane with one __match_any_sync among themselves.
    for (int r = 0; r < Rw; r++) {
        const int blk = w * Rw + r;
        if (blk >= nblk) break;
        const int p = 32 * blk + lane;
        const bool valid = p < P;
        uint32_t b = 0, c0 = 0, w4 = 0;
        if (valid) {
            uint32_t hp;
            w4 = sf_ldsu(c.sdb + p);
            b = sf_bucket<NMAX>(w4, &hp);
            c0 = cnt16[4 * b + w];
        }
        __syncwarp();
        if (valid) atomicAdd(&cnt32[2 * b + fsel], inc);
        __syncwarp();
        uint32_t m = 0;
        if (valid) m = (uint32_t)cnt16[4 * b + w] - c0;
        const bool multi = valid && m > 1;
        const uint32_t cm = __ballot_sync(FULL_MASK, multi);
        uint32_t cl = 0;
        if (multi) {
            const uint32_t peers = __match_any_sync(cm, b);
            cl = __popc(peers & ((1u << lane) - 1u));
        }
        if (valid) c.ord[c0 + cl] = (uint16_t)((uint32_t)p | (SfOrd<NMAX>::fp(w4 >> 24) << SfOrd<NMAX>::POSB));
    }
    __syncthreads();
    SF_PH(12);
    // first position per trigram hash (the counters are dead now): fo32 in A, then a u16 copy behind mlen / mpos
    // for the parse (c.fo16) and the literal filter has3
    uint32_t *fo = (uint32_t *)c.A;
    static_assert(C::NB * 4 <= 2 * NMAX, "fo32 must end before the bitmaps");
    for (int i = tid; i < C::NB / 4; i += SF_T) ((uint4 *)fo)[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
    for (int i = tid; i < 6 * C::NWORDS; i += SF_T) c.has3[i] = 0; // has3 | eval | vis | vis2 | ism | lenhi
    __syncthreads();
    for (int blk = w; blk < nblk; blk += SF_W) {
        const int p = 32 * blk + lane;
        if (p < P) atomicMin(&fo[((sf_ldsu(c.sdb + p) & 0xFFFFFFu) * 2654435761u) >> (32 - C::HB)], (uint32_t)p);
    }
    __syncthreads();
    for (int blk = w; blk < nblk; blk += SF_W) {
        const int p = 32 * blk + lane;
        bool has = false;
        if (p < P) has = fo[((sf_ldsu(c.sdb + p) & 0xFFFFFFu) * 2654435761u) >> (32 - C::HB)] < (uint32_t)p;
        const uint32_t hw = __ballot_sync(FULL_MASK, has);
        if (lane == 0) c.has3[blk] = hw;
    }
    uint16_t *fo16 = c.fo16();
    for (int i = tid; i < C::NB; i += SF_T) fo16[i] = (uint16_t)min(fo[i], 0xFFFFu);
    __syncthreads();
    SF_PH(16);
}

// Longest match for the positions p of the groups with need == true (earliest among the longest, capped at
// min(32, n - p): compression_methods.py:283-313); warp-uniform.  The candidates of the (up to four) positions a
// warp evaluates at once are pooled: item j of the warp = entry k of the bucket of owner o, 32 items per step with
// every lane busy, the owner's maximum is kept by a shared atomicMax on len << 16 | (0xFFFF - pos) -- which is the
// reference's "first strictly longer match".  (One group per bucket, 8 entries per step, cost the longest of the
// four buckets for all of them: 365 warp instructions per call, ncu.)
// Returns the key, or 0 when no match of >= 3 bytes exists.
template <int NMAX> __device__ __forceinline__ uint32_t sf_evaluate(const SfCtx<NMAX> &c, int p, bool need)
{
    constexpr int NO = 32 / SF_G;                       // owners (chains) per warp
    const int n = c.n, lane = threadIdx.x & 31;
    const int sub = lane & (SF_G - 1), g = lane / SF_G;
    uint32_t *ws = c.wsc + (threadIdx.x >> 5) * SF_WSW; // rec[NO][8] | best[NO] | first3[NO] | prefix[NO + 1]
    uint32_t *wbest = ws + 8 * NO, *wf3 = wbest + NO;
    const uint32_t pa = c.sdb + (need ? p : 0);
    const uint32_t wp0 = sf_ldsu(pa);
    const int cap = min(32, n - p);
    uint32_t hp;
    const uint32_t own = sf_bucket<NMAX>(wp0, &hp);
    // (A) matches of >= 4 bytes: the entries of p's own bucket
    int i0 = 0, cA = 0;
    if (need) { // the entries before p (ascending: lower bound of p in its bucket)
        i0 = (int)sf_lds16(c.bstb + 2 * own);
        int lo = i0, hi = (int)sf_lds16(c.bstb + 2 * own + 2);
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if ((int)(sf_lds16(c.ordb + 2 * mid) & SfOrd<NMAX>::POSMASK) < p) lo = mid + 1; else hi = mid;
        }
        cA = lo - i0;
    }
    if (sub == 0) {
        ws[8 * g + 0] = (uint32_t)p;
        ws[8 * g + 2] = wp0;
        ws[8 * g + 3] = (uint32_t)cap | (SfOrd<NMAX>::fp(wp0 >> 24) << 8);
        wbest[g] = 0;
        wf3[g] = 0xFFFFu;
        if (need) SF_COUNT(30, 1);
    }
    // An owner contributes at most SF_ROUND entries per round, in ascending order, and leaves as soon as its best
    // reaches the cap: nothing behind an entry that matches the whole look-ahead can be earlier.  (Periodic data
    // puts half of the chunk into one bucket; without the rounds every token looked at all of it: 3.5 GB/s.)
    int done_items = 0; // entries of this owner's bucket already looked at
    while (__any_sync(FULL_MASK, done_items < cA)) {
        const int cR = min(cA - done_items, SF_ROUND);
        int M;
        int pre[NO]; // exclusive prefix of the owners' item counts, in registers (it was 7 shared loads per item)
        {   // (lane SF_G * o holds owner o's count)
            const int v = sub == 0 ? cR : 0;
            const int inc = warp_incl_scan(v);
            M = __shfl_sync(FULL_MASK, inc, 31);
#pragma unroll
            for (int t = 0; t < NO; t++) pre[t] = __shfl_sync(FULL_MASK, inc - v, t * SF_G);
            if (sub == 0) ws[8 * g + 1] = (uint32_t)(i0 + done_items);
        }
        __syncwarp();
        for (int base = 0; base < M; base += 32) {
            const int j = base + lane;
            int o = 0, pb = 0;
#pragma unroll
            for (int t = 1; t < NO; t++) { const bool ge = j >= pre[t]; o += ge; pb = ge ? pre[t] : pb; }
            const int k = j - pb;
            __syncwarp();
            const uint32_t cur = wbest[o]; // best of the steps before this one
            __syncwarp();
            if (lane == 0) SF_COUNT(31, 1);
            if (j < M) {
                const int po = (int)ws[8 * o + 0];
                const uint32_t capfp = ws[8 * o + 3];
                const int capo = (int)(capfp & 0xFFu);
                const int bl = (int)(cur >> 16);
                if (bl < capo) {
                    const uint32_t e = sf_lds16(c.ordb + 2 * ((int)ws[8 * o + 1] + k));
                    const int q = (int)(e & SfOrd<NMAX>::POSMASK);
                    bool cand = (e >> SfOrd<NMAX>::POSB) == (capfp >> 8);
                    if (NMAX > 4096) cand = cand && (q + 4096 >= po); // window_size (compression_methods.py:294)
                    // with a match in hand only a strictly longer one counts (later entries are later positions)
                    if (cand && bl >= 4) cand = sf_lds8(c.sdb + q + bl) == sf_lds8(c.sdb + po + bl);
                    if (cand) {
                        const uint32_t qa = c.sdb + q, pao = c.sdb + po;
                        const uint32_t qab = qa & ~3u, qsh = (qa & 3u) * 8, pab = pao & ~3u, psh = (pao & 3u) * 8;
                        uint32_t qlo = sf_lds32(qab + 4);
                        uint32_t x = __funnelshift_r(sf_lds32(qab), qlo, qsh) ^ ws[8 * o + 2];
                        if (x == 0) {
                            int len = 32;
                            uint32_t plo = sf_lds32(pab + 4);
#pragma unroll 1
                            for (int kk = 1; kk < 8; kk++) {
                                if (4 * kk >= capo) break; // (the rest lies beyond the look-ahead)
                                const uint32_t qhi = sf_lds32(qab + 4 * kk + 4), phi = sf_lds32(pab + 4 * kk + 4);
                                x = __funnelshift_r(qlo, qhi, qsh) ^ __funnelshift_r(plo, phi, psh);
                                SF_COUNT(32, 1);
                                if (x) { len = 4 * kk + ((__ffs(x) - 1) >> 3); break; }
                                qlo = qhi; plo = phi;
                            }
                            len = min(len, capo);
                            atomicMax(&wbest[o], ((uint32_t)len << 16) | (uint32_t)(0xFFFF - q));
                        }
                    }
                }
            }
        }
        __syncwarp();
        done_items += cR;
        if ((int)(wbest[g] >> 16) >= cap) done_items = cA; // this owner is done
        __syncwarp();
    }
    __syncwarp();
    uint32_t best = wbest[g];
    // (B) no match of >= 4 bytes: the earliest earlier position with the same 3 bytes
    bool needB = need && (best >> 16) < 4;
    if (needB) { // fast path: the first position with p's trigram hash carries p's trigram -> it is the answer
        const uint32_t f = c.fo16()[hp >> (32 - SfCfg<NMAX>::HB)];
        if ((NMAX <= 4096 || (int)f + 4096 >= p) && ((sf_ldsu(c.sdb + f) ^ wp0) & 0xFFFFFFu) == 0) {
            best = (3u << 16) | (0xFFFFu - f); // (f < p: has3 was set)
            needB = false;
        }
    }
    if (__any_sync(FULL_MASK, needB)) {
        // it lies in one of the 8 buckets of the class, which are adjacent in ord
        int j0 = 0, cB = 0;
        if (needB) {
            j0 = (int)sf_lds16(c.bstb + 2 * (own & ~7u));
            cB = (int)sf_lds16(c.bstb + 2 * (own & ~7u) + 16) - j0;
        }
        __syncwarp();
        const int v = sub == 0 ? cB : 0;
        const int inc = warp_incl_scan(v);
        const int MB = __shfl_sync(FULL_MASK, inc, 31);
        int pre[NO];
#pragma unroll
        for (int t = 0; t < NO; t++) pre[t] = __shfl_sync(FULL_MASK, inc - v, t * SF_G);
        if (sub == 0) ws[8 * g + 4] = (uint32_t)j0;
        __syncwarp();
        for (int base = 0; base < MB; base += 32) {
            const int j = base + lane;
            if (lane == 0) SF_COUNT(39, 1);
            if (j < MB) {
                int o = 0, pb = 0;
#pragma unroll
                for (int t = 1; t < NO; t++) { const bool ge = j >= pre[t]; o += ge; pb = ge ? pre[t] : pb; }
                const int k = j - pb;
                const int po = (int)ws[8 * o + 0];
                const int q = (int)(sf_lds16(c.ordb + 2 * ((int)ws[8 * o + 4] + k)) & SfOrd<NMAX>::POSMASK);
                bool cand = q < po;
                if (NMAX > 4096) cand = cand && (q + 4096 >= po);
                if (cand && ((sf_ldsu(c.sdb + q) ^ ws[8 * o + 2]) & 0xFFFFFFu) == 0) atomicMin(&wf3[o], (uint32_t)q);
            }
        }
        __syncwarp();
        const uint32_t q3 = wf3[g];
        if (needB && q3 != 0xFFFFu) best = (3u << 16) | (0xFFFFu - q3);
    }
    return best;
}

// ---- Dictionary: lazy match evaluation ---------------------------------------------------------------
// All chains of a warp advance in lockstep: every loop below is warp-uniform (full-mask votes and shuffles), a
// chain = a group of SF_G lanes that share p and take the same branches.  (A first version ran each group in its
// own while loop with group masks: the groups drifted apart and the warp issued every group's path separately,
// 11 of 32 lanes active, ncu.)
//
// One step of all chains: tokens from position p until the chain leaves [.., s1).  FIX = false: speculative
// chain of a segment (marks c.vis).  FIX = true: the true chain entering the segment at p; marks c.vis2 and stops
// as soon as it meets the speculative chain (result -1 - meeting position).  Otherwise result = exit position.
template <int NMAX, bool FIX>
__device__ __forceinline__ int sf_chains(SfCtx<NMAX> &c, int p, int s1, bool act)
{
    const int lane = threadIdx.x & 31;
    const int sub = lane & (SF_G - 1);
    uint32_t *mark = FIX ? c.vis2 : c.vis;
    uint16_t *mm16 = c.mm16();
    int result = p;
    act = act && p < s1;
    while (__any_sync(FULL_MASK, act)) {
        if ((threadIdx.x & 31) == 0) SF_COUNT(FIX ? 34 : 33, 1);
        if (sub == 0 && act) SF_COUNT(FIX ? 36 : 35, 1);
        // (1) literals: everything before the next position whose trigram hash occurred earlier
        if (act) {
            int nx;
            {
                int wd = p >> 5;
                uint32_t hw = c.has3[wd] & (0xFFFFFFFFu << (p & 31));
                for (;;) {
                    if (hw) { nx = 32 * wd + __ffs(hw) - 1; break; }
                    wd++;
                    if (32 * wd >= s1) { nx = s1; break; }
                    hw = c.has3[wd];
                }
                nx = min(nx, s1);
            }
            if (nx > p) {
                int lim = nx;
                if (FIX) { // does the speculative chain visit one of the literals [p, nx)?
                    int wd = p >> 5;
                    uint32_t vw = c.vis[wd] & (0xFFFFFFFFu << (p & 31));
                    for (;;) {
                        if (vw) { lim = min(nx, 32 * wd + __ffs(vw) - 1); break; }
                        wd++;
                        if (32 * wd >= nx) break;
                        vw = c.vis[wd];
                    }
                }
                for (int wd = (p >> 5) + sub; 32 * wd < lim; wd += SF_G) { // set bits [p, lim): one word per lane
                    const int lo = max(p, 32 * wd) & 31, hi = min(lim, 32 * wd + 32) - 32 * wd;
                    mark[wd] |= (hi >= 32 ? 0xFFFFFFFFu : ((1u << hi) - 1u)) & (0xFFFFFFFFu << lo);
                }
                if (FIX && lim < nx) { result = -1 - lim; act = false; }
                else {
                    p = nx;
                    if (p >= s1) { result = p; act = false; }
                }
            }
        }
        __syncwarp();
        // (2) the token at p
        const uint32_t bit = 1u << (p & 31);
        const int wd = p >> 5;
        int L = 0;
        bool need = false;
        if (act) {
            if (FIX && (c.vis[wd] & bit)) { result = -1 - p; act = false; }
            else if (c.eval[wd] & bit) L = c.match_len(p);
            else need = true;
        }
        if (__any_sync(FULL_MASK, need)) {
            const uint32_t best = sf_evaluate<NMAX>(c, p, need);
            if (need) {
                L = (int)(best >> 16);
                if (sub == 0) {
                    c.eval[wd] |= bit;
                    if (L >= 3) {
                        const int q = (int)(0xFFFFu - (best & 0xFFFFu));
                        mm16[p] = (uint16_t)((uint32_t)(p - q - 1) | ((uint32_t)((L - 3) & 15) << 12));
                        c.ism[wd] |= bit;
                        if (L >= 19) c.lenhi[wd] |= bit;
                    }
                }
            }
        }
        if (act) {
            if (sub == 0) mark[wd] |= bit;
            p += L >= 3 ? L : 1;
            if (p >= s1) { result = p; act = false; }
        }
        __syncwarp();
    }
    return result;
}

// The true chain through [r0, r1) (multiples of 32, r1 may be n), entered at `entry` (r0 <= entry): the token
// starts go to c.vis2, *bytes = payload bytes of the tokens that start inside the range.  Returns the position
// at which the chain leaves the range.  Block-collective.
template <int NMAX> __device__ inline int sf_lz_parse_range(SfCtx<NMAX> &c, int r0, int r1, int entry, int *bytes_out)
{
    const int tid = threadIdx.x, lane = tid & 31;
    const int sub = lane & (SF_G - 1);
    // Segment of this group: consecutive segments go to different warps.  A position has the more candidates the
    // further back it lies in the chunk, and a warp pools the candidates of its chains, so with one contiguous
    // quarter of the chunk per warp the last warp did the most work and the first one waited at the barrier
    // (phase clocks: 20 % of the chunk time on log text, 36 % on binary records).
    constexpr int GPW = 32 / SF_G;
    const int grp = ((tid / SF_G) % GPW) * SF_W + (tid / SF_G) / GPW;
    if (entry >= r1) { *bytes_out = 0; return entry; }
    const int seg = max(32, ((((r1 - r0) + SF_NG - 1) / SF_NG) + 31) & ~31);
    const int s0 = r0 + grp * seg, s1 = min(r1, s0 + seg);
    const int start = grp == 0 ? entry : s0;
    const int last = (r1 - r0 - 1) / seg; // last group with a segment
    int *gspec = c.gst, *gcur = c.gst + SF_NG, *gdone = c.gst + 2 * SF_NG, *gmerge = c.gst + 3 * SF_NG;
    SF_PH_DECL
    // speculative chains
    const int ex = sf_chains<NMAX, false>(c, start, s1, s0 < r1);
    if (sub == 0) { gspec[grp] = ex; gcur[grp] = ex; gdone[grp] = start; gmerge[grp] = s0; }
    SF_PH(13);
    __syncthreads();
    SF_PH(14);
    // stitch: the true chain enters segment g where the true chain of segment g - 1 left it
    for (int round = 0; round < SF_NG; round++) {
        const int e = grp == 0 ? entry : gcur[grp - 1];
        const bool redo = s0 < r1 && grp > 0 && e != gdone[grp];
        __syncthreads(); // every gcur has been read
        if (threadIdx.x == 0) SF_COUNT(37, 1);
        if (sub == 0 && redo) SF_COUNT(38, 1);
        if (__any_sync(FULL_MASK, redo)) {
            if (redo)
                for (int wd = (s0 >> 5) + sub; 32 * wd < s1; wd += SF_G) c.vis2[wd] = 0;
            __syncwarp();
            const int x = sf_chains<NMAX, true>(c, e, s1, redo && e < s1);
            if (redo && sub == 0) {
                int cur, mg;
                if (e >= s1) { cur = e; mg = s1; }
                else if (x < 0) { mg = -1 - x; cur = gspec[grp]; }
                else { mg = s1; cur = x; }
                gcur[grp] = cur; gmerge[grp] = mg; gdone[grp] = e;
            }
        }
        if (!__syncthreads_or(redo)) break;
    }
    SF_PH(15);
    // token starts of the true chain: vis2 | (vis at or behind the meeting point)
    int bytes = 0;
    for (int wd = (r0 >> 5) + tid; 32 * wd < r1; wd += SF_T) {
        const int g = (32 * wd - r0) / seg;
        const int mg = gmerge[g];
        uint32_t keep;
        if (mg <= 32 * wd) keep = 0xFFFFFFFFu;
        else if (mg >= 32 * wd + 32) keep = 0;
        else keep = 0xFFFFFFFFu << (mg - 32 * wd);
        const uint32_t reach = c.vis2[wd] | (c.vis[wd] & keep);
        bytes += 2 * __popc(reach) + 2 * __popc(reach & c.ism[wd]);
        c.vis2[wd] = reach;
    }
    const int exitp = gcur[last];
    *bytes_out = sf_block_sum(bytes, c.red); // (its barriers also keep gcur alive until everybody has read it)
    return exitp;
}

// Exact Dictionary payload length of the chunk, or SF_ABORTED as soon as the exact cost of a prefix plus the
// smallest possible cost of the rest (4 bytes per 32) reaches `cutoff` (staged == true: the chunk is parsed in
// three stages; a speed gamble for chunks whose Dictionary payload is expected to lose, never a change of the
// outcome).  Afterwards c.vis2 holds the token-start bitmap of the true chain, c.ism marks the match tokens,
// mlen / mpos hold their lengths and sources.  Requires sf_lz_index.
#define SF_ABORTED 0x7fffffff
template <int NMAX> __device__ inline int sf_lz_parse(SfCtx<NMAX> &c, int cutoff, bool staged)
{
    const int n = c.n;
    int bound[4] = {0, n, n, n};
    int nst = 1;
    if (staged && n >= 1024) { nst = 3; bound[1] = (11 * n / 32) & ~31; bound[2] = (9 * n / 16) & ~31; }
    int entry = 0, total = 0;
    for (int st = 0; st < nst; st++) {
        int bytes;
        entry = sf_lz_parse_range<NMAX>(c, bound[st], bound[st + 1], entry, &bytes);
        total += bytes;
        if (st + 1 < nst) {
            const int rest = n - entry;
            const int lb = total + (rest > 0 ? 4 * (rest >> 5) + min(4, 2 * (rest & 31)) : 0);
            if (lb >= cutoff) return SF_ABORTED;
        }
    }
    return total;
}


// Dictionary payload -> c.pay (after sf_lz_parse; ord is dead by now)
template <int NMAX> __device__ inline void sf_lz_emit(SfCtx<NMAX> &c)
{
    using C = SfCfg<NMAX>;
    const int n = c.n, tid = threadIdx.x;
    const int nw = (n + 31) >> 5;
    const int wpt = (nw + SF_T - 1) / SF_T; // words per thread, contiguous
    int bytes = 0;
    for (int wd = tid * wpt; wd < min(nw, (tid + 1) * wpt); wd++) {
        const uint32_t reach = c.vis2[wd];
        bytes += 2 * __popc(reach) + 2 * __popc(reach & c.ism[wd]);
    }
    int total;
    int off = sf_block_excl_scan(bytes, c.red, &total);
    uint16_t *pay16 = (uint16_t *)c.pay; // token offsets are even
    const uint16_t *mm16 = c.mm16();
    for (int wd = tid * wpt; wd < min(nw, (tid + 1) * wpt); wd++) {
        uint32_t reach = c.vis2[wd];
        const uint32_t mm = c.ism[wd];
        while (reach) {
            const int bit = __ffs(reach) - 1;
            reach &= reach - 1;
            const int p = 32 * wd + bit;
            if ((mm >> bit) & 1u) {
                if (off + 4 <= C::PAY_BYTES) {
                    const uint32_t v = mm16[p];
                    const int d = (int)(v & 0xFFFu) + 1;
                    const int L = 3 + (int)(v >> 12) + (((c.lenhi[wd] >> bit) & 1u) ? 16 : 0);
                    pay16[off >> 1] = (uint16_t)(1u | ((uint32_t)(d & 0xFF) << 8));
                    pay16[(off >> 1) + 1] = (uint16_t)((uint32_t)(d >> 8) | ((uint32_t)L << 8));
                }
                off += 4;
            } else {
                if (off + 2 <= C::PAY_BYTES) pay16[off >> 1] = (uint16_t)((uint32_t)c.sd[p] << 8);
                off += 2;
            }
        }
    }
    __syncthreads();
}

// A lower bound of the Dictionary payload that needs no index and no parse (tokens: a literal costs 2 bytes, a match
// of >= 3 bytes 4 bytes, compression_methods.py:211-231).
//   * Let D be the number of distinct 4-grams of the chunk, i.e. of positions whose 4-gram has no earlier
//     occurrence ("first" positions).  Inside a match the 4-gram of every position but the last three is a copy of
//     an earlier one, so a first position is covered by a literal or by one of the last three bytes of a match.
//   * Let F be the number of positions p whose trigram and the trigrams at p - 1 and p - 2 all occur for the first
//     time.  Such a position is a literal in every parse: a match that covers p would contain the whole trigram
//     at p, at p - 1 or at p - 2.  These positions are first positions of their 4-gram as well.
//   Hence D - F <= other literals + 3 * matches, and the payload is at least 2 F + 4/3 (D - F) = (4 D + 2 F) / 3.
// On the bench corpus: low-cardinality chunks 3 187 bytes from D alone (Huffman payload 1 599), CSV 2 038 + 196
// (Huffman 2 037), text 772 + 107 (Huffman 2 043: no help there).  D is counted with a 17-bit hash set and the
// first trigram positions come from a 12-bit hash table of minimum positions; both can only lose some, and the
// bound grows with D and F.  `need`: the bound is only compared with this value (F is skipped when D suffices).
// Uses region A and the first words of the ord / payload area (free between the Huffman build and the index).
// Block-collective.
template <int NMAX> __device__ inline int sf_lz_bound_ngrams(SfCtx<NMAX> &c, int need)
{
    static_assert(SfCfg<NMAX>::A_BYTES >= 16384, "hash set / table fit region A");
    const int n = c.n, tid = threadIdx.x, lane = tid & 31;
    uint32_t *bm = (uint32_t *)c.A; // 2^17 bits
    for (int i = tid; i < 1024; i += SF_T) ((uint4 *)bm)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    for (int p = tid; p < n - 3; p += SF_T) {
        const uint32_t h = (sf_ldsu(c.sdb + p) * 2654435761u) >> 15;
        atomicOr(&bm[h >> 5], 1u << (h & 31));
    }
    __syncthreads();
    int cnt = 0;
    for (int i = tid; i < 4096; i += SF_T) cnt += __popc(bm[i]);
    const int D = sf_block_sum(cnt, c.red);
    if ((4 * D) / 3 >= need) return (4 * D) / 3;
    // first position per trigram hash, then the bitmap of first positions
    uint32_t *fo = (uint32_t *)c.A;          // 4096 entries
    uint32_t *fw = (uint32_t *)c.ord;        // NMAX / 32 words
    __syncthreads();
    for (int i = tid; i < 1024; i += SF_T) ((uint4 *)fo)[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
    __syncthreads();
    for (int p = tid; p < n - 2; p += SF_T)
        atomicMin(&fo[((sf_ldsu(c.sdb + p) & 0xFFFFFFu) * 2654435761u) >> 20], (uint32_t)p);
    __syncthreads();
    for (int p0 = 32 * (tid >> 5); p0 < n; p0 += SF_T) { // a warp per 32 positions
        const int p = p0 + lane;
        bool first = false;
        if (p < n - 2) first = fo[((sf_ldsu(c.sdb + p) & 0xFFFFFFu) * 2654435761u) >> 20] == (uint32_t)p;
        const uint32_t w = __ballot_sync(FULL_MASK, first);
        if (lane == 0) fw[p0 >> 5] = w;
    }
    __syncthreads();
    int forced = 0;
    for (int wd = tid; 32 * wd < n - 3; wd += SF_T) {
        const uint32_t f = fw[wd], fp = wd ? fw[wd - 1] : 0u;
        uint32_t z = f & ((f << 1) | (fp >> 31)) & ((f << 2) | (fp >> 30));
        if (n - 3 < 32 * wd + 32) z &= 0xFFFFFFFFu >> (32 * wd + 32 - (n - 3)); // positions with a 4-gram only
        forced += __popc(z);
    }
    const int F = sf_block_sum(forced, c.red);
    return (4 * D + 2 * F) / 3;
}

// ---- the decision ------------------------------------------------------------------------------------
struct SfOut { int type; int len; };

// size-range eligibility (adaptive_compressor.py:114-127, tested on the clamped size :565-567)
__device__ __forceinline__ bool sf_eligible(int id, int n)
{
    switch (id) {
    case 1: return n >= 32 && n <= 4096;
    case 2: return n >= 128 && n <= 8192;
    case 3: return n >= 32 && n <= 8192;
    case 4: return n >= 32 && n <= 4096;
    }
    return false;
}

// Evaluate the chunk staged by sf_load; the winner's payload is left in c.pay.  The outcome is the reference's
// (methods in id order, the first strictly smaller payload wins, benefit test len + ovh < n); the order of
// evaluation is not: a trial is skipped when its payload provably cannot end up as the winner.
template <int NMAX> __device__ SfOut sf_select(SfCtx<NMAX> &c, uint32_t mask, int ovh)
{
    const int n = c.n;
    SfOut o;
    o.type = 255; o.len = n;
    const bool rle_el = (mask & 2u) && sf_eligible(1, n);
    const bool lz_el = (mask & 4u) && sf_eligible(2, n) && n >= 100;
    const bool hf_el = (mask & 8u) && sf_eligible(3, n) && n >= 100;
    // Delta (id 4) always produces n bytes, so (n + overhead) / n > 1 never wins (adaptive_compressor.py:574-577).
    if (!rle_el && !lz_el && !hf_el) return o;

    SF_PH_DECL
    int best_type = 255, best_len = 0x7fffffff;
    if (rle_el) {
        int pairs;
        if (sf_rle_features(c, &pairs)) {
            const int len = 2 * pairs;
            if (len + ovh < n) { best_type = 1; best_len = len; }
        }
    }
    SF_PH(1);
    // smallest payloads the other two methods can produce: RLE at or below both wins outright
    const int lz_min = lz_el ? sf_lz_lower_bound(n) : 0x7fffffff;
    const int hf_min = hf_el ? 1 + 5 * 2 + 4 + ((n + 7) >> 3) : 0x7fffffff;
    if (best_type == 1 && best_len <= lz_min && best_len <= hf_min) {
        sf_rle_emit(c);
        o.type = 1; o.len = best_len;
        return o;
    }
    if (lz_el || hf_el) {
        SfStats st;
        sf_stats(c, lz_el, st);
        SF_PH(2);
        SfHuff hs = sf_huff_scratch(c);
        // gates (compression_methods.py:315-343, 551-574); the quotient distinct / s < 0.8 as an exact integer compare
        const bool lz_ok = lz_el && 10 * st.distinct3 < 8 * min(1000, n);
        bool hf_ok = hf_el && st.K >= 2 && st.K <= 255;
        if (hf_ok) {
            if (fabsf(st.H - 7.0f) < 0.02f) { // near the threshold: fp64, in the reference's summation order
                sf_first_order(c, hs, st.K);
                hf_ok = sf_entropy_ordered(c, hs, st.K) < 7.0;
            } else hf_ok = st.H < 7.0f;
        }
        int hf_len = 0x7fffffff, hf_bits = 0;
        if (hf_ok) {
            // entropy lower bound (st.H is within 3e-4 of the entropy): bits >= max(n, n * H)
            const int lb = 1 + 5 * st.K + 4 + (int)ceilf(fmaxf((float)n, (float)n * (st.H - 0.002f) - 0.01f) * 0.125f);
            if (lb < best_len && lb + ovh < n) {
                hf_bits = sf_huff_build(c, hs, st.K);
                const int len = 1 + 5 * st.K + 4 + ((hf_bits + 7) >> 3);
                if (len < best_len && len + ovh < n) hf_len = len;
            }
        }
        SF_PH(3);
        if (lz_ok) {
            // the Dictionary payload wins iff it is < the RLE payload, <= the Huffman payload and beneficial
            int cutoff = min(best_len, n - ovh);
            if (hf_len != 0x7fffffff) cutoff = min(cutoff, hf_len + 1);
            // many distinct trigrams and a Huffman payload in hand: the Dictionary payload usually loses clearly
            const bool staged = hf_len != 0x7fffffff && 100 * st.distinct3 >= 34 * min(1000, n);
            // ... and often provably, before any index or parse (sf_lz_bound_ngrams: every low-cardinality and CSV chunk
            // of the bench corpus)
            bool hopeless = false;
            if (lz_min < cutoff && staged) hopeless = sf_lz_bound_ngrams(c, cutoff) >= cutoff;
            if (lz_min < cutoff && !hopeless) {
                sf_lz_index(c);
                SF_PH(4);
                const int len = sf_lz_parse(c, cutoff, staged);
                SF_PH(5);
                if (len < cutoff) {
                    sf_lz_emit(c);
                    SF_PH(6);
                    o.type = 2; o.len = len;
                    return o;
                }
            }
        }
        if (hf_len != 0x7fffffff) { // (already known to beat RLE and to be beneficial)
            __syncthreads();
            sf_huff_emit(c, hs, st.K, hf_bits);
            SF_PH(7);
            o.type = 3; o.len = hf_len;
            return o;
        }
    }
    if (best_type == 1) {
        sf_rle_emit(c);
        o.type = 1; o.len = best_len;
    }
    return o;
}
