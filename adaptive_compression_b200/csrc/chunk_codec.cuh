// chunk_codec.cuh -- per-chunk device code: should_use gates and the four native encoders.
// One CTA (AMBC_BLOCK threads) works on one chunk staged in shared memory.  Every function
// here is block-collective: all threads of the CTA must call it with the same arguments.
//
// Reference behaviour restated (file:line relative to the reference repo):
//   RLE        compression_methods.py:78-114, gate :154-180
//   Dictionary compression_methods.py:195-234 + 283-313 (earliest-longest greedy LZ77), gate :315-343
//   Huffman    compression_methods.py:354-405 + 472-549 ((weight, leader) tie-break), gate :551-574
//   Delta      compression_methods.py:585-608, gate :640-667
#pragma once
#include "common.cuh"

struct ChunkCtx {
    uint8_t *sd;       // chunk bytes, 16-byte aligned, followed by AMBC_PAD zero bytes
    int n;             // chunk length (<= AMBC_NMAX)
    uint8_t *pay;      // payload buffer, 16-byte aligned
    int pcap;          // payload capacity; longer payloads are counted but not stored
    uint16_t *sorted;  // n+2 entries (LZ bucket-sorted positions); reused as Huffman bit words
    uint16_t *bstart;  // AMBC_NBUCKET+1 bucket starts
    uint8_t *X;        // 16 KiB + 64 scratch (LZ counters / trigram set / block exits / Huffman nodes)
    uint8_t *mlen;     // n match lengths (0 = literal)
    uint16_t *mpos;    // n match positions
    uint32_t *hist;    // 256 byte counts
    uint32_t *bmask;   // run-boundary bitmap, ceil(n/32) words
    uint32_t *reach;   // token-start bitmap, ceil(n/32) words
    uint8_t *estart;   // per 32-block chain entry offset
    int *red;          // 32 ints of reduction scratch (8-byte aligned)
    // names-based match search (lz_names.cuh), chunks of at most LZ2_NMAX bytes
    uint32_t *T;       // LZ2_TSLOTS hash slots (32 KiB)
    uint16_t *nameA;   // LZ2_NMAX first-occurrence names (two buffers, alternating levels)
    uint16_t *nameB;
    uint8_t *L;        // LZ2_LBYTES of list memory: participant / item lists and the slot memo
    // Huffman code table by symbol; survives the Dictionary trial (the rest of the Huffman scratch does not)
    uint32_t *hcode;   // [256]
    uint8_t *hlen;     // [256]
};
#define AMBC_HTAB_BYTES 1280

#define LZ2_NMAX 4096
#define LZ2_TSLOTS 8192
#define LZ2_LBYTES 32768
#define LZ2_BYTES (LZ2_TSLOTS * 4 + 2 * LZ2_NMAX * 2 + LZ2_LBYTES)

// scratch region X: LZ per-warp bucket counters, or 16 KiB for the other users
#define AMBC_XBYTES ((AMBC_WARPS * AMBC_NBUCKET * 2) > 16384 ? (AMBC_WARPS * AMBC_NBUCKET * 2) : 16384)
#define AMBC_BPT (AMBC_NBUCKET / AMBC_BLOCK) // buckets per thread in the counter scan
static_assert(AMBC_BPT >= 2 && AMBC_BPT % 2 == 0 && AMBC_BPT * AMBC_BLOCK == AMBC_NBUCKET, "bucket scan layout");

// shared-memory bytes of a ChunkCtx for chunk size N and payload capacity pcap
__host__ __device__ inline size_t r16(size_t x) { return (x + 15) & ~(size_t)15; }
__host__ __device__ inline size_t chunkctx_smem_bytes(int N, int pcap)
{
    size_t sorted_b = 2 * (size_t)(N + 2);
    if (sorted_b < (size_t)pcap + 16) sorted_b = (size_t)pcap + 16;
    size_t nb = (size_t)(N + 31) / 32;
    return r16((size_t)N) + AMBC_PAD          // sd
           + r16((size_t)pcap) + 16           // pay
           + r16(sorted_b)                    // sorted
           + r16(2 * (AMBC_NBUCKET + 1))      // bstart
           + AMBC_XBYTES + 64                 // X
           + r16((size_t)N)                   // mlen
           + r16(2 * (size_t)N)               // mpos
           + 1024                             // hist
           + r16(nb * 4) * 2                  // bmask, reach
           + r16(nb)                          // estart
           + 128                              // red
           + AMBC_HTAB_BYTES                  // hcode, hlen
           + LZ2_BYTES;                       // T, nameA, nameB, fol
}

__device__ inline void chunkctx_carve(ChunkCtx &c, uint8_t *base, int N, int pcap)
{
    size_t sorted_b = 2 * (size_t)(N + 2);
    if (sorted_b < (size_t)pcap + 16) sorted_b = (size_t)pcap + 16;
    size_t nb = (size_t)(N + 31) / 32;
    uint8_t *p = base;
    c.sd = p; p += r16((size_t)N) + AMBC_PAD;
    c.pay = p; p += r16((size_t)pcap) + 16;
    c.sorted = (uint16_t *)p; p += r16(sorted_b);
    c.bstart = (uint16_t *)p; p += r16(2 * (AMBC_NBUCKET + 1));
    c.X = p; p += AMBC_XBYTES + 64;
    c.mlen = p; p += r16((size_t)N);
    c.mpos = (uint16_t *)p; p += r16(2 * (size_t)N);
    c.hist = (uint32_t *)p; p += 1024;
    c.bmask = (uint32_t *)p; p += r16(nb * 4);
    c.reach = (uint32_t *)p; p += r16(nb * 4);
    c.estart = p; p += r16(nb);
    c.red = (int *)p; p += 128;
    c.hcode = (uint32_t *)p; c.hlen = p + 1024; p += AMBC_HTAB_BYTES;
    c.T = (uint32_t *)p; p += LZ2_TSLOTS * 4;
    c.nameA = (uint16_t *)p; p += LZ2_NMAX * 2;
    c.nameB = (uint16_t *)p; p += LZ2_NMAX * 2;
    c.L = p;
    c.pcap = pcap;
    c.n = 0;
}

// Stage chunk [src, src+n) in c.sd and zero the pad.  Ends with __syncthreads().
__device__ inline void chunk_load(ChunkCtx &c, const uint8_t *__restrict__ src, int n)
{
    c.n = n;
    copy_g2s(c.sd, src, n);
    int padend = (int)r16((size_t)n) + AMBC_PAD;
    for (int i = n + threadIdx.x; i < padend; i += AMBC_BLOCK) c.sd[i] = 0;
    __syncthreads();
}

// ---------------------------------------------------------------------------------------
// features: histogram, run-boundary bitmap, sampled gates, distinct trigrams, entropy
// ---------------------------------------------------------------------------------------
struct ChunkFeatures {
    int rep;        // sampled adjacent-equal count      (compression_methods.py:172-175)
    int small;      // sampled |delta| < 32 count        (:658-662)
    int distinct3;  // distinct trigrams among the first min(n-3, 1000) positions (:333-336)
    int K;          // distinct byte values
    int rle_pairs;  // (byte,count) pairs RLE would emit -- defined only when the RLE gate holds
    float H;        // entropy in fp32 (|error| < 3e-4): decides the Huffman gate away from 7.0 and bounds its size;
                    // near 7.0 the caller sums in fp64 in the reference's order (chunk_entropy_ordered)
};

// extract byte j (compile-time after unrolling) of a 32-byte slice held in two uint4
__device__ __forceinline__ uint32_t slice_byte(const uint4 &a, const uint4 &b, int j)
{
    uint32_t w;
    switch (j >> 2) {
    case 0: w = a.x; break; case 1: w = a.y; break; case 2: w = a.z; break; case 3: w = a.w; break;
    case 4: w = b.x; break; case 5: w = b.y; break; case 6: w = b.z; break; default: w = b.w; break;
    }
    return (w >> ((j & 3) * 8)) & 0xFF;
}

__device__ inline void chunk_features(ChunkCtx &c, ChunkFeatures &f)
{
    const int n = c.n, tid = threadIdx.x;
    const int nsl = (n + 31) >> 5;
    uint32_t *tri = (uint32_t *)c.X; // 2048-slot open-addressing set
    for (int i = tid; i < 256; i += AMBC_BLOCK) c.hist[i] = 0;
    for (int i = tid; i < 2048 / 4; i += AMBC_BLOCK) ((uint4 *)tri)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();

    // histogram (run-aggregated shared atomics) + run-boundary bitmap
    for (int s = tid; s < nsl; s += AMBC_BLOCK) {
        const uint4 a = *(const uint4 *)(c.sd + 32 * s);
        const uint4 b = *(const uint4 *)(c.sd + 32 * s + 16);
        const int m = min(32, n - 32 * s);
        uint32_t prev = s ? c.sd[32 * s - 1] : 0x100u; // 0x100: never equal -> boundary at position 0
        uint32_t mask = 0, cur = 0, cnt = 0;
#pragma unroll
        for (int j = 0; j < 32; j++) {
            if (j < m) {
                uint32_t v = slice_byte(a, b, j);
                if (v != prev) mask |= 1u << j;
                if (j == 0) { cur = v; cnt = 1; }
                else if (v == cur) cnt++;
                else { atomicAdd(&c.hist[cur], cnt); cur = v; cnt = 1; }
                prev = v;
            }
        }
        atomicAdd(&c.hist[cur], cnt);
        c.bmask[s] = mask;
    }

    // sampled gates: RLE (:165-180) and Delta (:651-667) share the sample positions
    int rep = 0, small = 0;
    if (n >= 4) {
        const int ss = min(1000, n);
        const int step = n < 2000 ? 1 : n / 1000; // == max(1, n // ss); constant divisor instead of a runtime division in every thread
        for (int i = tid * step; i < n - 1; i += AMBC_BLOCK * step) {
            int x = c.sd[i], y = c.sd[i + 1];
            rep += (x == y);
            small += (abs(x - y) < 32);
        }
    }
    // distinct trigrams (:326-343)
    int ins = 0;
    if (n >= 100) {
        const int cnt3 = min(n - 3, min(1000, n));
        for (int i = tid; i < cnt3; i += AMBC_BLOCK) {
            uint32_t t = lds_u32u(c.sd + i) & 0xFFFFFFu;
            uint32_t key = t + 1, h = (t * 2654435761u) >> 21;
            for (;;) {
                uint32_t old = atomicCAS(&tri[h], 0u, key);
                if (old == 0u) { ins++; break; }
                if (old == key) break;
                h = (h + 1) & 2047;
            }
        }
    }
    // one block reduction for the three gate counters (also orders hist / bmask writes before the reads below)
    int *redx = (int *)(c.X + 8192); // 4 x AMBC_WARPS ints behind the trigram set
    {
        const int lane = tid & 31, w = tid >> 5;
        int a = warp_sum(rep), b = warp_sum(small), d = warp_sum(ins);
        if (lane == 0) { redx[w] = a; redx[AMBC_WARPS + w] = b; redx[2 * AMBC_WARPS + w] = d; }
        __syncthreads();
        f.rep = warp_sum(lane < AMBC_WARPS ? redx[lane] : 0);
        f.small = warp_sum(lane < AMBC_WARPS ? redx[AMBC_WARPS + lane] : 0);
        f.distinct3 = warp_sum(lane < AMBC_WARPS ? redx[2 * AMBC_WARPS + lane] : 0);
        __syncthreads();
    }

    // RLE pair count: a run of R bytes -> ceil(R/255) pairs (:95-109).  Only needed (and only
    // defined) when the RLE gate holds (:177-180), which is rare outside run-heavy data.
    int pairs = 0;
    const bool rle_gate = n >= 4 && 10 * f.rep > 3 * (min(1000, n) - 1); // == rep / (s - 1) > 0.3 in fp64
    if (rle_gate) {
        for (int s = tid; s < nsl; s += AMBC_BLOCK) {
            uint32_t w = c.bmask[s];
            while (w) {
                int bit = __ffs(w) - 1;
                w &= w - 1;
                int p = 32 * s + bit, q;
                if (w) q = 32 * s + __ffs(w) - 1;
                else {
                    q = n;
                    for (int s2 = s + 1; s2 < nsl; s2++) {
                        uint32_t w2 = c.bmask[s2];
                        if (w2) { q = 32 * s2 + __ffs(w2) - 1; break; }
                    }
                }
                const int R = q - p;
                pairs += R <= 255 ? 1 : (R + 254) / 255;
            }
        }
    }

    // entropy (:566-574) in fp32; the caller resolves near-threshold cases in fp64, in the reference's order
    float hsum = 0.0f;
    int k = 0;
    const float inv_n = 1.0f / (float)n;
    for (int b = tid; b < 256; b += AMBC_BLOCK) {
        uint32_t cnt = c.hist[b];
        if (cnt) {
            k++;
            const float p = (float)cnt * inv_n;
            hsum -= p * __log2f(p);
        }
    }
    {   // one block reduction for pairs, K and H
        const int lane = tid & 31, w = tid >> 5;
        int a = warp_sum(pairs), b = warp_sum(k);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) hsum += __shfl_xor_sync(FULL_MASK, hsum, d);
        float *redd = (float *)(redx + 2 * AMBC_WARPS);
        if (lane == 0) { redx[w] = a; redx[AMBC_WARPS + w] = b; redd[w] = hsum; }
        __syncthreads();
        float rh = lane < AMBC_WARPS ? redd[lane] : 0.0f;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) rh += __shfl_xor_sync(FULL_MASK, rh, d); // (xor tree: the same sum in every lane)
        f.rle_pairs = warp_sum(lane < AMBC_WARPS ? redx[lane] : 0);
        f.K = warp_sum(lane < AMBC_WARPS ? redx[AMBC_WARPS + lane] : 0);
        f.H = rh;
        __syncthreads();
    }
}

// first-occurrence order of the byte values (Counter insertion order, :368-370 / :566).
// order[r] = r-th distinct byte value; firstpos scratch = 256 uint32.  Collective.
// Ranks of the present entries of keys[256] (absent = 0xFFFFFFFF, present keys distinct): the
// present keys are compacted first, so the all-pairs compare costs K^2 instead of 256^2.
// emit(rank, symbol, key) runs once per present entry.  Scratch (see huff_scratch): ck[256],
// cs[256], cw[8].  Block-collective, three __syncthreads().  Returns K.
template <class F>
__device__ __forceinline__ int rank_present(const uint32_t *keys, uint32_t *ck, uint8_t *cs, int *cw, F emit)
{
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    uint32_t key = 0xFFFFFFFFu;
    if (tid < 256) key = keys[tid];
    const uint32_t m = __ballot_sync(FULL_MASK, key != 0xFFFFFFFFu);
    if (tid < 256 && lane == 0) cw[w] = __popc(m);
    __syncthreads();
    int base = 0, K = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { const int x = cw[i]; if (i < w) base += x; K += x; }
    if (key != 0xFFFFFFFFu) {
        const int at = base + __popc(m & ((1u << lane) - 1));
        ck[at] = key;
        cs[at] = (uint8_t)tid;
    }
    __syncthreads();
    if (tid < K) {
        const uint32_t k = ck[tid];
        int r = 0;
        for (int j = 0; j < K; j++) r += (ck[j] < k);
        emit(r, (int)cs[tid], k);
    }
    __syncthreads();
    return K;
}

__device__ inline void chunk_first_order(ChunkCtx &c, uint32_t *firstpos, uint8_t *order)
{
    const int n = c.n, tid = threadIdx.x;
    for (int i = tid; i < 256; i += AMBC_BLOCK) firstpos[i] = 0xFFFFFFFFu;
    __syncthreads();
    volatile uint32_t *fpv = firstpos;
    for (int s = tid; 8 * s < n; s += AMBC_BLOCK) { // 8 bytes per thread and step
        const uint2 w = *(const uint2 *)(c.sd + 8 * s);
        const int m = min(8, n - 8 * s);
        uint32_t prev = 0x100u;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const uint32_t v = ((j < 4 ? w.x : w.y) >> (8 * (j & 3))) & 0xFFu;
            // values only decrease, so a stale plain read can only cause a redundant atomic
            if (j < m && v != prev && fpv[v] > (uint32_t)(8 * s + j)) atomicMin(&firstpos[v], (uint32_t)(8 * s + j));
            prev = v;
        }
    }
    __syncthreads();
    rank_present(firstpos, (uint32_t *)(c.X + 3072), c.X + 8448, (int *)(c.X + 8704),
                 [&](int r, int sym, uint32_t) { order[r] = (uint8_t)sym; });
}

// exact Python-order entropy: e -= p*log2(p) over the Counter's insertion order, no FMA
// contraction.  Result valid in every thread.  Collective.
__device__ inline double chunk_entropy_ordered(ChunkCtx &c, int K, const uint8_t *order)
{
    volatile double *out = (volatile double *)c.red;
    if (threadIdx.x == 0) {
        double e = 0.0;
        for (int r = 0; r < K; r++) {
            double p = __ddiv_rn((double)c.hist[order[r]], (double)c.n);
            e = __dsub_rn(e, __dmul_rn(p, log2(p)));
        }
        out[0] = e;
    }
    __syncthreads();
    double e = out[0];
    __syncthreads();
    return e;
}

// ---------------------------------------------------------------------------------------
// RLE encode (compression_methods.py:78-114): payload -> c.pay.  Returns the length.
// Requires c.bmask from chunk_features.  Collective.
// ---------------------------------------------------------------------------------------
__device__ inline int chunk_rle_encode(ChunkCtx &c)
{
    const int n = c.n, tid = threadIdx.x;
    const int nsl = (n + 31) >> 5;
    const int spt = (nsl + AMBC_BLOCK - 1) / AMBC_BLOCK; // slices per thread, contiguous
    int pairs = 0;
    for (int s = tid * spt; s < min(nsl, (tid + 1) * spt); s++) {
        uint32_t w = c.bmask[s];
        while (w) {
            int bit = __ffs(w) - 1;
            w &= w - 1;
            int p = 32 * s + bit, q;
            if (w) q = 32 * s + __ffs(w) - 1;
            else {
                q = n;
                for (int s2 = s + 1; s2 < nsl; s2++) {
                    uint32_t w2 = c.bmask[s2];
                    if (w2) { q = 32 * s2 + __ffs(w2) - 1; break; }
                }
            }
            pairs += (q - p + 254) / 255;
        }
    }
    int total;
    int off = 2 * block_excl_scan(pairs, c.red, &total);
    for (int s = tid * spt; s < min(nsl, (tid + 1) * spt); s++) {
        uint32_t w = c.bmask[s];
        while (w) {
            int bit = __ffs(w) - 1;
            w &= w - 1;
            int p = 32 * s + bit, q;
            if (w) q = 32 * s + __ffs(w) - 1;
            else {
                q = n;
                for (int s2 = s + 1; s2 < nsl; s2++) {
                    uint32_t w2 = c.bmask[s2];
                    if (w2) { q = 32 * s2 + __ffs(w2) - 1; break; }
                }
            }
            int R = q - p;
            uint8_t v = c.sd[p];
            while (R > 0) {
                int cnt = R > 255 ? 255 : R;
                if (off + 2 <= c.pcap) { c.pay[off] = v; c.pay[off + 1] = (uint8_t)cnt; }
                off += 2;
                R -= cnt;
            }
        }
    }
    __syncthreads();
    return 2 * total;
}

// ---------------------------------------------------------------------------------------
// Delta encode (compression_methods.py:585-608): payload -> c.pay (needs pcap >= n).
// ---------------------------------------------------------------------------------------
__device__ inline int chunk_delta_encode(ChunkCtx &c)
{
    const int n = c.n;
    for (int i = threadIdx.x; i < n; i += AMBC_BLOCK) {
        uint8_t v = i ? (uint8_t)(c.sd[i] - c.sd[i - 1]) : c.sd[0];
        if (i < c.pcap) c.pay[i] = v;
    }
    __syncthreads();
    return n;
}

// ---------------------------------------------------------------------------------------
// Dictionary / greedy LZ77 (compression_methods.py:195-234, 283-313)
// ---------------------------------------------------------------------------------------
// Levels of the top-down match search: n-gram lengths, ascending.  A position is searched in
// the bucket of its LZ_LEVELS[k]-gram only if no earlier position shares its
// LZ_LEVELS[k+1]-gram, so its longest match is at most LZ_LEVELS[k+1]-1 bytes and the ascending
// scan can stop at the first candidate of that length.  Any level set starting at 3 is exact;
// the set only changes how many candidates are visited.
#define LZ_MAX_LEVELS 8
static __device__ __constant__ int LZ_LEVELS[LZ_MAX_LEVELS] = {3, 4, 6, 10, 0, 0, 0, 0};
static __device__ __constant__ int LZ_NLEVELS = 4;
static __device__ __constant__ int LZ_COOP_T = 24; // buckets with more candidates are scanned by a whole warp
static __device__ __constant__ int LZ_FORCE_BUCKETS = 0; // test knob: always use the bucket search
static inline int lz_force_buckets_upload(int on)
{
    return cudaMemcpyToSymbol(LZ_FORCE_BUCKETS, &on, sizeof on) == cudaSuccess ? 0 : -1;
}

// hash of the L-gram at shared-memory address s (L <= 16)
__device__ __forceinline__ uint32_t lz_hash_l(const uint8_t *s, int L)
{
    uintptr_t a = (uintptr_t)s;
    const uint32_t *w = (const uint32_t *)(a & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(a & 3) * 8;
    uint32_t w0 = w[0], w1 = w[1];
    uint32_t x = __funnelshift_r(w0, w1, sh);
    if (L < 4) return ((x & 0xFFFFFFu) * 2654435761u) >> (32 - AMBC_HB);
    uint32_t h = x * 2654435761u;
    int rem = L - 4, k = 1;
    while (rem > 0) {
        uint32_t w2 = w[k + 1];
        x = __funnelshift_r(w1, w2, sh);
        if (rem < 4) x &= (1u << (8 * rem)) - 1;
        h = (h ^ (h >> 15) ^ x) * 2246822519u;
        w1 = w2; k++; rem -= 4;
    }
    return (h ^ (h >> 13)) * 3266489917u >> (32 - AMBC_HB);
}

// Stable bucket sort of positions [0, P) by the hash of their L-gram: c.sorted (ascending
// positions inside each bucket) and c.bstart.  Uses c.X as [AMBC_WARPS][AMBC_NBUCKET] counters.
// Collective.
__device__ inline void lz_bucket_sort(ChunkCtx &c, int P, int L)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    uint16_t *cnt = (uint16_t *)c.X;
    for (int i = tid; i < AMBC_WARPS * AMBC_NBUCKET * 2 / 16; i += AMBC_BLOCK)
        ((uint4 *)cnt)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    const int Q = ((P + AMBC_BLOCK - 1) / AMBC_BLOCK) * 32; // positions per warp
    const int wbeg = wid * Q, wend = min(P, wbeg + Q);
    uint16_t *mycnt = cnt + wid * AMBC_NBUCKET;
    for (int base = wbeg; base < wend; base += 32) { // pass 1: per-warp bucket counts
        int p = base + lane;
        bool valid = p < wend;
        uint32_t h = valid ? lz_hash_l(c.sd + p, L) : (uint32_t)(AMBC_NBUCKET + lane);
        uint32_t peers = __match_any_sync(FULL_MASK, h);
        uint32_t prior = valid ? mycnt[h] : 0;
        __syncwarp();
        if (valid && lane == 31 - __clz(peers)) mycnt[h] = (uint16_t)(prior + __popc(peers));
        __syncwarp();
    }
    __syncthreads();
    {   // exclusive scan in (bucket-major, warp-minor) order; thread owns AMBC_BPT buckets
        constexpr int NW = AMBC_BPT / 2; // 32-bit words (two u16 counters) per warp row
        uint32_t v[AMBC_WARPS][NW];
#pragma unroll
        for (int w = 0; w < AMBC_WARPS; w++) {
            const uint32_t *src = (const uint32_t *)(cnt + w * AMBC_NBUCKET + AMBC_BPT * tid);
#pragma unroll
            for (int k = 0; k < NW; k++) v[w][k] = src[k];
        }
        uint32_t run = 0;
#pragma unroll
        for (int hh = 0; hh < AMBC_BPT; hh++) {
#pragma unroll
            for (int w = 0; w < AMBC_WARPS; w++) {
                uint32_t word = v[w][hh >> 1];
                uint32_t x = (hh & 1) ? (word >> 16) : (word & 0xFFFF);
                v[w][hh >> 1] = (hh & 1) ? ((word & 0xFFFF) | (run << 16)) : ((word & 0xFFFF0000u) | run);
                run += x;
            }
        }
        int tot;
        uint32_t off = (uint32_t)block_excl_scan((int)run, c.red, &tot);
        uint32_t off2 = off | (off << 16);
#pragma unroll
        for (int w = 0; w < AMBC_WARPS; w++) {
            uint32_t *dst = (uint32_t *)(cnt + w * AMBC_NBUCKET + AMBC_BPT * tid);
#pragma unroll
            for (int k = 0; k < NW; k++) { v[w][k] += off2; dst[k] = v[w][k]; }
        }
        uint32_t *bs = (uint32_t *)(c.bstart + AMBC_BPT * tid);
#pragma unroll
        for (int k = 0; k < NW; k++) bs[k] = v[0][k];
        if (tid == 0) c.bstart[AMBC_NBUCKET] = (uint16_t)P;
    }
    __syncthreads();
    for (int base = wbeg; base < wend; base += 32) { // pass 2: ordered scatter
        int p = base + lane;
        bool valid = p < wend;
        uint32_t h = valid ? lz_hash_l(c.sd + p, L) : (uint32_t)(AMBC_NBUCKET + lane);
        uint32_t peers = __match_any_sync(FULL_MASK, h);
        uint32_t prior = valid ? mycnt[h] : 0;
        __syncwarp();
        if (valid) {
            c.sorted[prior + __popc(peers & ((1u << lane) - 1))] = (uint16_t)p;
            if (lane == 31 - __clz(peers)) mycnt[h] = (uint16_t)(prior + __popc(peers));
        }
        __syncwarp();
    }
    __syncthreads();
}


// common-prefix length (bytes, up to 4*nw) of the data at shared address s with the words pw[]
__device__ __forceinline__ int lz_match_len(const uint8_t *s, const uint32_t (&pw)[8], int nw)
{
    uintptr_t a = (uintptr_t)s;
    const uint32_t *w = (const uint32_t *)(a & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(a & 3) * 8;
    uint32_t lo_w = w[0];
    int len = 4 * nw;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        if (k < nw) {
            uint32_t hi_w = w[k + 1];
            uint32_t x = __funnelshift_r(lo_w, hi_w, sh) ^ pw[k];
            if (x) { len = 4 * k + ((__ffs(x) - 1) >> 3); break; }
            lo_w = hi_w;
        }
    }
    return len;
}

#include "lz_names.cuh"

// Earliest-longest match for every position by scanning n-gram buckets (any chunk size up to
// AMBC_NMAX; honours the 4096-byte window).  c.mlen must be zero.  Collective.
#ifdef V_NOINLINE_BUCKETS
__device__ __noinline__ void lz_match_all_buckets(ChunkCtx &c)
#else
__device__ inline void lz_match_all_buckets(ChunkCtx &c)
#endif
{
    const int n = c.n, tid = threadIdx.x, lane = tid & 31;
    // ---- earliest-longest match for every position, longest n-gram level first -----------
    for (int li = LZ_NLEVELS - 1; li >= 0; li--) {
        const int L = LZ_LEVELS[li];
        const int U = (li == LZ_NLEVELS - 1) ? 32 : LZ_LEVELS[li + 1] - 1;
        const int P = n - L + 1; // positions that have a whole L-gram
        if (P < 2) continue;
        lz_bucket_sort(c, P, L);
        const int nwU = (U + 3) >> 2;
        // deferred queue for long buckets (scanned warp-cooperatively below): slots as u16 in c.pay
        uint16_t *defq = (uint16_t *)c.pay;
        const int qcap = c.pcap >> 1;
        volatile int *qn = c.red + 28, *qhead = c.red + 29;
        if (tid == 0) { *qn = 0; *qhead = 0; }
        __syncthreads();
        const int Pr = (P + 31) & ~31; // whole warps iterate together (ballot below)
        for (int s = tid; s < Pr; s += AMBC_BLOCK) {
            int p = 0, b0 = 0;
            bool todo = false;
            if (s < P) {
                p = c.sorted[s];
                if (!c.mlen[p]) { // not resolved at a longer level
                    b0 = c.bstart[lz_hash_l(c.sd + p, L)];
                    todo = b0 < s;
                }
            }
            bool defer = todo && (s - b0 > LZ_COOP_T);
            uint32_t dmask = __ballot_sync(FULL_MASK, defer);
            if (dmask) {
                int base = 0;
                if (lane == 0) base = atomicAdd((int *)qn, __popc(dmask));
                base = __shfl_sync(FULL_MASK, base, 0);
                int slot = base + __popc(dmask & ((1u << lane) - 1));
                if (defer) {
                    if (slot < qcap) defq[slot] = (uint16_t)s;
                    else defer = false; // queue full: scan it here
                }
            }
            if (!todo || defer) continue;
            const int cap = min(U, n - p); // lookahead_size 32 / end of data (:295, :304-305)
            uint32_t pw[8];
            {
                uintptr_t a = (uintptr_t)(c.sd + p);
                const uint32_t *w = (const uint32_t *)(a & ~(uintptr_t)3);
                const uint32_t sh = (uint32_t)(a & 3) * 8;
                uint32_t lo_w = w[0];
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    if (k < nwU) { uint32_t hi_w = w[k + 1]; pw[k] = __funnelshift_r(lo_w, hi_w, sh); lo_w = hi_w; }
                    else pw[k] = 0;
                }
            }
            const int lo = p - 4096; // window_size (:294)
            int best = 0, bpos = 0;
            for (int j = b0; j < s; j++) {
                const int i = c.sorted[j];
                if (i < lo) continue;
                int len = lz_match_len(c.sd + i, pw, nwU);
                len = min(len, cap);
                if (len >= L && len > best) { // a true L-gram match, strictly longer (:309-311)
                    best = len; bpos = i;
                    if (len == cap) break;
                }
            }
            if (best) { c.mlen[p] = (uint8_t)best; c.mpos[p] = (uint16_t)bpos; }
        }
        __syncthreads();
        // long buckets: one warp per slot, 32 candidates per step, ascending, same tie rule
        const int nq = min(*qn, qcap);
        for (;;) {
            int q = 0;
            if (lane == 0) q = atomicAdd((int *)qhead, 1);
            q = __shfl_sync(FULL_MASK, q, 0);
            if (q >= nq) break;
            const int s = defq[q];
            const int p = c.sorted[s];
            const int b0 = c.bstart[lz_hash_l(c.sd + p, L)];
            const int cap = min(U, n - p);
            uint32_t pw[8];
            {
                uintptr_t a = (uintptr_t)(c.sd + p);
                const uint32_t *w = (const uint32_t *)(a & ~(uintptr_t)3);
                const uint32_t sh = (uint32_t)(a & 3) * 8;
                uint32_t lo_w = w[0];
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    if (k < nwU) { uint32_t hi_w = w[k + 1]; pw[k] = __funnelshift_r(lo_w, hi_w, sh); lo_w = hi_w; }
                    else pw[k] = 0;
                }
            }
            const int lo = p - 4096;
            int best = 0, bpos = 0;
            for (int base = b0; base < s; base += 32) {
                const int j = base + lane;
                int i = 0, len = 0;
                if (j < s) {
                    i = c.sorted[j];
                    if (i >= lo) {
                        len = min(lz_match_len(c.sd + i, pw, nwU), cap);
                        if (len < L) len = 0;
                    }
                }
                const int m = __reduce_max_sync(FULL_MASK, len);
                if (m > best) { // the earliest candidate of the new maximum: lowest lane
                    const int first = __ffs(__ballot_sync(FULL_MASK, len == m)) - 1;
                    best = m;
                    bpos = __shfl_sync(FULL_MASK, i, first);
                    if (best == cap) break;
                }
            }
            if (lane == 0 && best) { c.mlen[p] = (uint8_t)best; c.mpos[p] = (uint16_t)bpos; }
        }
        __syncthreads();
    }
}

__device__ __forceinline__ void lz_zero_mlen(ChunkCtx &c)
{
    for (int p = threadIdx.x * 16; p < (int)r16((size_t)c.n); p += AMBC_BLOCK * 16)
        *(uint4 *)(c.mlen + p) = make_uint4(0, 0, 0, 0);
    __syncthreads();
}

// Payload -> c.pay (as far as pcap allows).  Returns the exact payload length.  Collective.
__device__ inline int chunk_lz_encode(ChunkCtx &c)
{
    const int n = c.n, tid = threadIdx.x;
    lz_zero_mlen(c);
    bool done = false;
    if (n <= LZ2_NMAX && !LZ_FORCE_BUCKETS) {
        done = lz2_match_all(c) == 0;
        if (!done) lz_zero_mlen(c); // a table overflowed (pathological key skew): redo with the bucket search
    }
    if (!done) lz_match_all_buckets(c);
    __syncthreads();

    // ---- token chain: pos -> pos + (len>2 ? len : 1) (:211-232), resolved per 32-block ---
    const int nb = (n + 31) >> 5;
    uint8_t *fexit = c.X; // fexit[q * nb + b]: where a chain entering block b at offset q leaves it
    for (int b = tid; b < nb; b += AMBC_BLOCK) {
        const uint4 a4 = *(const uint4 *)(c.mlen + 32 * b);
        const uint4 b4 = *(const uint4 *)(c.mlen + 32 * b + 16);
#pragma unroll
        for (int q = 31; q >= 0; q--) {
            uint32_t L = slice_byte(a4, b4, q);
            int t = q + (L >= 3 ? (int)L : 1);
            uint8_t fx;
            if (32 * b + q >= n) fx = 255; // past the end of the chunk
            else if (t >= 32) fx = (uint8_t)(t - 32);
            else fx = fexit[t * nb + b];
            fexit[q * nb + b] = fx;
        }
    }
    __syncthreads();
    {   // entry offset of every block on the chain from position 0: groups of 32 blocks are composed
        // for all 32 entry offsets at once (one warp per group, lane = entry offset), then the few
        // groups are chained and every group is walked from its true entry
        uint8_t *gexit = c.X + 8192 + 2048; // [group][entry offset]
        uint8_t *gentry = gexit + 256;      // entry offset of each group
        const int ng = (nb + 31) >> 5, wid = tid >> 5, lane = tid & 31;
        if (wid < ng) {
            int e = lane;
            const int bend = min(nb, 32 * wid + 32);
            for (int b = 32 * wid; b < bend; b++)
                if (e != 255) e = fexit[e * nb + b];
            gexit[32 * wid + lane] = (uint8_t)e;
        }
        __syncthreads();
        if (tid == 0) {
            int e = 0;
            for (int g = 0; g < ng; g++) {
                gentry[g] = (uint8_t)e;
                if (e != 255) e = gexit[32 * g + e];
            }
        }
        __syncthreads();
        if (tid < ng) {
            int e = gentry[tid];
            const int bend = min(nb, 32 * tid + 32);
            for (int b = 32 * tid; b < bend; b++) {
                c.estart[b] = (uint8_t)e;
                if (e != 255) e = fexit[e * nb + b];
            }
        }
    }
    __syncthreads();
    // per block: token-start mask, match mask, payload bytes; then every position emits its own token
    uint32_t *mmask = (uint32_t *)(c.X + 8192);        // behind fexit (32 * nb <= 8 KiB)
    uint32_t *boff = (uint32_t *)(c.X + 8192 + 1024);  // payload offset of the block's first token
    const int bpt = (nb + AMBC_BLOCK - 1) / AMBC_BLOCK; // blocks per thread, contiguous
    int tbytes = 0;
    for (int b = tid * bpt; b < min(nb, (tid + 1) * bpt); b++) {
        int q = c.estart[b];
        uint32_t mask = 0, mm = 0;
        boff[b] = (uint32_t)tbytes; // relative to this thread's first block until the scan below
        while (q < 32 && 32 * b + q < n) {
            mask |= 1u << q;
            int L = c.mlen[32 * b + q];
            if (L >= 3) { mm |= 1u << q; tbytes += 4; q += L; } else { tbytes += 2; q += 1; }
        }
        c.reach[b] = mask;
        mmask[b] = mm;
    }
    int total;
    const int off0 = block_excl_scan(tbytes, c.red, &total);
    for (int b = tid * bpt; b < min(nb, (tid + 1) * bpt); b++) boff[b] += (uint32_t)off0;
    __syncthreads();
    uint16_t *pay16 = (uint16_t *)c.pay; // token offsets are even
    for (int p = tid; p < n; p += AMBC_BLOCK) {
        const int b = p >> 5;
        const uint32_t bit = 1u << (p & 31), R = c.reach[b];
        if (R & bit) {
            const uint32_t below = R & (bit - 1), mm = mmask[b];
            const int off = (int)boff[b] + 2 * __popc(below) + 2 * __popc(below & mm);
            if (mm & bit) {
                if (off + 4 <= c.pcap) {
                    const int d = p - (int)c.mpos[p];
                    pay16[off >> 1] = (uint16_t)(1u | ((uint32_t)(d & 0xFF) << 8));
                    pay16[(off >> 1) + 1] = (uint16_t)((uint32_t)(d >> 8) | ((uint32_t)c.mlen[p] << 8));
                }
            } else if (off + 2 <= c.pcap) pay16[off >> 1] = (uint16_t)((uint32_t)c.sd[p] << 8);
        }
    }
    __syncthreads();
    return total;
}

// ---------------------------------------------------------------------------------------
// Huffman (compression_methods.py:354-405, 472-549)
// ---------------------------------------------------------------------------------------
// scratch layout inside c.X
struct HuffScratch {
    uint32_t *key;      // [256] (count << 8 | sym) or 0xFFFFFFFF
    uint32_t *nodeW;    // [512]
    uint16_t *lead;     // [512]
    uint16_t *parent;   // [512]
    uint8_t *nbit;      // [512]
    uint8_t *lenOf;     // [256] by symbol
    uint8_t *order;     // [256] first-occurrence order
    uint32_t *codeOf;   // [256] by symbol
    uint32_t *firstpos; // [256]
    uint8_t *leafsym;   // [256] symbol of sorted leaf j
};
__device__ inline HuffScratch huff_scratch(ChunkCtx &c)
{
    HuffScratch h;
    uint8_t *X = c.X;
    h.key = (uint32_t *)X;
    h.nodeW = (uint32_t *)(X + 1024);
    h.lead = (uint16_t *)(X + 3072);
    h.parent = (uint16_t *)(X + 4096);
    h.nbit = X + 5120;
    h.lenOf = c.hlen;
    h.order = X + 5888;
    h.codeOf = c.hcode;
    h.firstpos = (uint32_t *)(X + 7168);
    h.leafsym = X + 8192;
    return h;
}

// Build the reference's tree for the counts in c.hist (K distinct values, 2 <= K <= 256):
// repeatedly merge the two smallest nodes under (weight, leader); lo gets bit 0, hi bit 1;
// leader(merged) = leader(lo) (:482-494).  Leaves are pre-sorted by (weight, symbol) and the
// merged nodes come out already ordered by the same key, so two queues suffice.
// Fills lenOf / codeOf and returns the total number of code bits.  Collective.
__device__ inline int chunk_huff_build(ChunkCtx &c, HuffScratch &h, int K)
{
    const int tid = threadIdx.x;
    for (int b = tid; b < 256; b += AMBC_BLOCK) {
        uint32_t cnt = c.hist[b];
        h.key[b] = cnt ? ((cnt << 8) | (uint32_t)b) : 0xFFFFFFFFu;
        h.lenOf[b] = 0;
        h.codeOf[b] = 0;
    }
    __syncthreads();
    // rank sort: keys are distinct; one word (weight << 8 | leader) orders nodes by (weight, leader)
    rank_present(h.key, (uint32_t *)(c.X + 3072), c.X + 8448, (int *)(c.X + 8704),
                 [&](int r, int sym, uint32_t k) { h.nodeW[r] = k; h.leafsym[r] = (uint8_t)sym; });
    __syncthreads();
    if (tid == 0) {
        // two-queue merge, both queue heads cached in registers: one reload per pick.  Weights stay
        // below 2^24 (chunks of at most 8192 bytes), leaders are byte values.
        int li = 0, mi = K, t = K;
        uint32_t kl = h.nodeW[0];      // head of the leaf queue
        uint32_t km = 0xFFFFFFFFu;     // head of the merged queue (empty)
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
            // merged weight = sum, leader = leader of the lower node (:482-494)
            const uint32_t nk = (((pk[0] >> 8) + (pk[1] >> 8)) << 8) | (pk[0] & 0xFFu);
            h.nodeW[t] = nk;
            h.parent[pick[0]] = (uint16_t)t; h.nbit[pick[0]] = 0;
            h.parent[pick[1]] = (uint16_t)t; h.nbit[pick[1]] = 1;
            if (mi == t) km = nk; // the merged queue was empty: the new node is its head
            t++;
        }
    }
    __syncthreads();
    const int root = 2 * K - 2;
    int bits = 0;
    for (int j = tid; j < K; j += AMBC_BLOCK) {
        int node = j, len = 0;
        uint32_t code = 0;
        while (node != root) {
            code |= (uint32_t)h.nbit[node] << len;
            len++;
            node = h.parent[node];
        }
        int sym = h.leafsym[j];
        h.lenOf[sym] = (uint8_t)len;
        h.codeOf[sym] = code;
        bits += len * (int)c.hist[sym];
    }
    return block_sum(bits, c.red);
}

// Payload (table in first-occurrence order + bit count + MSB-first bit stream, :379-403)
// -> c.pay.  Requires chunk_huff_build and c.bmask.  Returns the payload length.  Collective.
__device__ inline int chunk_huff_emit(ChunkCtx &c, HuffScratch &h, int K, int total_bits)
{
    const int n = c.n, tid = threadIdx.x;
    chunk_first_order(c, h.firstpos, h.order);
    const int hdr = 1 + 5 * K + 4;
    const int nbytes = (total_bits + 7) >> 3;
    if (tid == 0 && c.pcap >= 1) c.pay[0] = (uint8_t)K;
    for (int r = tid; r < K; r += AMBC_BLOCK) {
        int o = 1 + 5 * r;
        if (o + 5 <= c.pcap) {
            int sym = h.order[r];
            c.pay[o] = (uint8_t)sym;
            store_u32le(c.pay + o + 1, c.hist[sym]);
        }
    }
    if (tid == 0 && hdr <= c.pcap) store_u32le(c.pay + hdr - 4, (uint32_t)total_bits);
    // bit stream built as big-endian 32-bit words in the (now dead) sorted[] region
    uint32_t *bw = (uint32_t *)c.sorted;
    const int nwords = (total_bits + 31) >> 5;
    const int wcap = min(nwords, (c.pcap >> 2) + 1);
    for (int i = tid; i < wcap; i += AMBC_BLOCK) bw[i] = 0;
    const int nsl = (n + 7) >> 3; // 8-byte slices, contiguous per thread
    const int spt = (nsl + AMBC_BLOCK - 1) / AMBC_BLOCK;
    int mybits = 0;
    for (int s = tid * spt; s < min(nsl, (tid + 1) * spt); s++) {
        const uint2 w = *(const uint2 *)(c.sd + 8 * s);
        const int m = min(8, n - 8 * s);
#pragma unroll
        for (int j = 0; j < 8; j++)
            if (j < m) mybits += h.lenOf[((j < 4 ? w.x : w.y) >> (8 * (j & 3))) & 0xFFu];
    }
    int tot;
    int g = block_excl_scan(mybits, c.red, &tot); // includes the barrier after zeroing bw
    {
        int w = g >> 5, used = g & 31;
        uint32_t cur = 0;
        for (int s = tid * spt; s < min(nsl, (tid + 1) * spt); s++) {
            const uint2 w8 = *(const uint2 *)(c.sd + 8 * s);
            const int m = min(8, n - 8 * s);
#pragma unroll
            for (int j = 0; j < 8; j++) {
                if (j >= m) break;
                const int sym = ((j < 4 ? w8.x : w8.y) >> (8 * (j & 3))) & 0xFFu;
                uint32_t code = h.codeOf[sym];
                int l = h.lenOf[sym];
                int space = 32 - used;
                if (l <= space) {
                    cur |= code << (space - l);
                    used += l;
                    if (used == 32) {
                        if (w < wcap) atomicOr(&bw[w], cur);
                        w++; cur = 0; used = 0;
                    }
                } else {
                    cur |= code >> (l - space);
                    if (w < wcap) atomicOr(&bw[w], cur);
                    w++;
                    used = l - space;
                    cur = code << (32 - used);
                }
            }
        }
        if (used && w < wcap) atomicOr(&bw[w], cur);
    }
    __syncthreads();
    for (int k = tid; k < nbytes; k += AMBC_BLOCK) {
        if (hdr + k < c.pcap) c.pay[hdr + k] = (uint8_t)(bw[k >> 2] >> (24 - 8 * (k & 3)));
    }
    __syncthreads();
    return hdr + nbytes;
}
