// lz_names.cuh -- exact earliest-longest match search of the Dictionary method for chunks of at
// most LZ2_NMAX bytes (the whole chunk lies inside window_size = 4096, compression_methods.py:187).
//
// The reference scans every earlier position i < p in ascending order and keeps the first
// strictly longer match, capped at min(32, n - p) (compression_methods.py:283-313).  So
//   mlen[p] = the largest L <= min(32, n - p) whose L-gram at p already occurred at some i < p, and
//   mpos[p] = the FIRST occurrence of that L-gram.
// Let name_L[p] = first position whose L-gram equals the one at p ("name"; name_L[p] == p: p is the
// head of its class).  Then mlen[p] = max { L : name_L[p] < p } and mpos[p] = name_mlen[p].
// Names are built without comparing strings:
//   name_4      hash of the 4 raw bytes (verified against the data),
//   name_3      only for heads of name_4 (a 4-byte match implies the 3-byte one),
//   name_2k     from the pair (name_k[p], name_k[p + k])                        (k = 4, 8, 16),
//   name_{k+j}  from the pair (name_k[p], name_k[p + j]), 0 < j < k, only for "participants":
//               heads at 2k whose k-gram occurs elsewhere (everybody else either has a match of
//               >= 2k bytes or no k-byte match at all).  The lengths of a bracket are visited in
//               binary-search order; a participant enters length m of the interval (lo, hi) only
//               if it is a head at hi and its lo-gram occurs elsewhere -- the first occurrence of
//               any m-gram that somebody matches always satisfies both.  Every round runs over a
//               dense item list that the previous round's resolve pass appended.
// Every "first occurrence of a key" is one open-addressing insert with atomicMin on the position;
// a later arrival at a key clears the slot's `single` bit ("this gram occurs more than once").
// Keys are verified through the name arrays, so the result is exact for any hash function.
// Names carry bit 15 = "the class has more than one member".
// Block-collective; returns false when a table overflowed (caller falls back to the bucket search).
#pragma once

#define LZ2_EMPTY 0xFFFFFFFFu
#define LZ2_GOLD 2654435761u
#define LZ2_NS 0x8000u           // name flag: the gram occurs at more than one position
#define LZ2_RSLOTS LZ2_TSLOTS     // table slots of a refinement pass
#define LZ2_RSHIFT 19            // 32 - log2(LZ2_RSLOTS)
#ifndef LZ2_PART_TARGET
#define LZ2_PART_TARGET 4096     // entries per refinement pass (load factor 1/2; measured best of 2048..4096)
#endif
#ifndef LZ2_BIN_MINK
#define LZ2_BIN_MINK 4           // smallest bracket refined in binary-search order (8: the (4,8) bracket uses the flat method)
#endif
#define LZ2_ISLOTS 8192          // slot memo entries

// slot value = tag << 14 | home << 13 | position << 1 | single: the claiming insert stores single = 1,
// every later arrival at the same key clears it (atomicMin with an even value, or atomicAnd).
// Pair tables hold their keys exactly: a table of 2^tbits slots takes keys below 2^W, W = tbits + 18;
// h = lz2_hash(key) is a bijection on W-bit values, its top tbits are the home slot and its low 18 bits the
// tag.  An entry that sits in its home slot (home = 1) is therefore identified by (slot, tag) alone -- no
// look at the names; only an entry displaced by linear probing (home = 0) is verified through the name
// arrays.  Keys that differ only above bit 23 (the node / length index) differ in the low 18 hash bits
// (the fold key ^= key >> 15 carries bits 24.. down to bits 9.., the odd multiply is a bijection on the
// low 18 bits), so that verification never confuses two nodes.
#define LZ2_HOME 0x2000u
__device__ __forceinline__ uint32_t lz2_hash(uint32_t key, uint32_t wmask)
{
    key ^= key >> 15;
    return (key * LZ2_GOLD) & wmask;
}
__device__ __forceinline__ void lz2_clear(ChunkCtx &c, int slots)
{
    for (int i = threadIdx.x * 4; i < slots; i += AMBC_BLOCK * 4)
        *(uint4 *)(c.T + i) = make_uint4(LZ2_EMPTY, LZ2_EMPTY, LZ2_EMPTY, LZ2_EMPTY);
}
__device__ __forceinline__ uint32_t lz2_slot_pos(uint32_t v) { return (v >> 1) & 0xFFFu; }
__device__ __forceinline__ uint32_t lz2_slot_name(uint32_t v) { return ((v >> 1) & 0xFFFu) | ((v & 1u) ? 0u : LZ2_NS); }

// first occurrence of the 4-byte gram `w` at p (32 key bits do not fit the exact scheme: verified against
// the data), table of LZ2_TSLOTS slots
__device__ __forceinline__ uint32_t lz2_insert_raw4(ChunkCtx &c, uint32_t w, int p)
{
    uint32_t s = (w * LZ2_GOLD) >> (32 - 13);
    const uint32_t val = ((uint32_t)p << 1) | 1u;
    for (;;) {
        const uint32_t q = atomicCAS(&c.T[s], LZ2_EMPTY, val);
        if (q == LZ2_EMPTY) return s;
        if (lds_u32u(c.sd + lz2_slot_pos(q)) == w) {
            if (val < q) atomicMin(&c.T[s], val & ~1u);
            else if (q & 1u) atomicAnd(&c.T[s], ~1u);
            return s;
        }
        s = (s + 1) & (LZ2_TSLOTS - 1);
    }
}

// first occurrence of the 3-byte gram `w` (< 2^24) at p: exact key as in the pair tables
__device__ __forceinline__ uint32_t lz2_insert_raw3(ChunkCtx &c, uint32_t w, int p, uint32_t mask, uint32_t wmask)
{
    const uint32_t h = lz2_hash(w, wmask);
    uint32_t s = h >> 18;
    uint32_t val = (h << 14) | LZ2_HOME | ((uint32_t)p << 1) | 1u;
    uint32_t q = atomicCAS(&c.T[s], LZ2_EMPTY, val);
    if (q == LZ2_EMPTY) return s;
    if ((q ^ val) < LZ2_HOME) {
        if (val < q) atomicMin(&c.T[s], val & ~1u);
        else if (q & 1u) atomicAnd(&c.T[s], ~1u);
        return s;
    }
    val &= ~LZ2_HOME;
    for (;;) { // the table is at most 1/4 full
        s = (s + 1) & mask;
        q = atomicCAS(&c.T[s], LZ2_EMPTY, val);
        if (q == LZ2_EMPTY) return s;
        if ((q ^ val) < LZ2_HOME && (lds_u32u(c.sd + lz2_slot_pos(q)) & 0xFFFFFFu) == w) {
            if (val < q) atomicMin(&c.T[s], val & ~1u);
            else if (q & 1u) atomicAnd(&c.T[s], ~1u);
            return s;
        }
    }
}

// first occurrence of the pair key with W-bit hash h (names S[p] = a, S[p + j] = b) in a table of
// (mask + 1) slots.  Returns the slot, or 0xFFFF and sets *overflow when the table is full.
__device__ __forceinline__ uint32_t lz2_insert_pair(ChunkCtx &c, uint32_t mask, uint32_t h, const uint16_t *S,
                                                    uint32_t a, uint32_t b, int p, int j, int *overflow)
{
    uint32_t s = h >> 18;
    uint32_t val = (h << 14) | LZ2_HOME | ((uint32_t)p << 1) | 1u;
    uint32_t q = atomicCAS(&c.T[s], LZ2_EMPTY, val);
    if (q == LZ2_EMPTY) return s;
    if ((q ^ val) < LZ2_HOME) { // same tag, at home: the same key
        if (val < q) atomicMin(&c.T[s], val & ~1u);
        else if (q & 1u) atomicAnd(&c.T[s], ~1u);
        return s;
    }
    val &= ~LZ2_HOME;
    for (uint32_t probes = 1; probes <= mask; probes++) {
        s = (s + 1) & mask;
        q = atomicCAS(&c.T[s], LZ2_EMPTY, val);
        if (q == LZ2_EMPTY) return s;
        if ((q ^ val) < LZ2_HOME) { // same tag, both displaced: the homes may differ
            const uint32_t qp = lz2_slot_pos(q);
            if (S[qp] == a && S[qp + j] == b) {
                if (val < q) atomicMin(&c.T[s], val & ~1u);
                else if (q & 1u) atomicAnd(&c.T[s], ~1u);
                return s;
            }
        }
    }
    *overflow = 1;
    return 0xFFFFu;
}

// name_4 (D) for every position, matches of length 4.  Returns "any match".
__device__ inline int lz2_level4(ChunkCtx &c, uint16_t *D)
{
    const int n = c.n, tid = threadIdx.x;
    lz2_clear(c, LZ2_TSLOTS);
    if (tid == 0) c.red[30] = 0; // level-3 list length
    __syncthreads();
    const int P = n - 3;
    for (int p = tid; p < n; p += AMBC_BLOCK) {
        uint32_t slot = 0xFFFFu;
        if (p < P) slot = lz2_insert_raw4(c, lds_u32u(c.sd + p), p);
        D[p] = (uint16_t)slot;
    }
    __syncthreads();
    // resolve; the heads (no 4-byte match) are listed for the 3-byte level
    uint16_t *list3 = (uint16_t *)c.L;
    volatile int *cnt = c.red + 30;
    const int lane = tid & 31;
    int nonhead = 0;
    for (int pb = 0; pb < n; pb += AMBC_BLOCK) {
        const int p = pb + tid;
        bool head3 = false;
        if (p < n) {
            const uint32_t slot = D[p];
            uint32_t nm = (uint32_t)p;
            if (slot != 0xFFFFu) nm = lz2_slot_name(c.T[slot]);
            D[p] = (uint16_t)nm;
            if ((nm & 0xFFFu) < (uint32_t)p) { c.mlen[p] = 4; c.mpos[p] = (uint16_t)(nm & 0xFFFu); nonhead++; }
            else head3 = p + 3 <= n; // (positions past n - 4 are their own name)
        }
        const uint32_t m = __ballot_sync(FULL_MASK, head3);
        if (m) {
            int base = 0;
            if (lane == 0) base = atomicAdd((int *)cnt, __popc(m));
            base = __shfl_sync(FULL_MASK, base, 0);
            if (head3) list3[base + __popc(m & ((1u << lane) - 1))] = (uint16_t)p;
        }
    }
    return __syncthreads_or(nonhead);
}

// matches of length exactly 3: only heads of name_4 can have one (listed by lz2_level4 in c.L).
// tmp: scratch buffer for the slots.
__device__ inline void lz2_level3(ChunkCtx &c, uint16_t *tmp)
{
    const int tid = threadIdx.x;
    const uint16_t *list3 = (const uint16_t *)c.L;
    const int cnt = c.red[30];
    const int tbits = min(13, max(10, 32 - __clz(max(4 * cnt, 2) - 1))); // table sized to the list (load <= 1/4)
    const uint32_t mask = (1u << tbits) - 1u, wmask = (1u << (tbits + 18)) - 1u;
    lz2_clear(c, 1 << tbits);
    __syncthreads();
    for (int i = tid; i < cnt; i += AMBC_BLOCK) {
        const int p = list3[i];
        tmp[i] = (uint16_t)lz2_insert_raw3(c, lds_u32u(c.sd + p) & 0xFFFFFFu, p, mask, wmask);
    }
    __syncthreads();
    for (int i = tid; i < cnt; i += AMBC_BLOCK) {
        const int p = list3[i];
        const uint32_t nm = lz2_slot_pos(c.T[tmp[i]]);
        if (nm < (uint32_t)p) { c.mlen[p] = 3; c.mpos[p] = (uint16_t)nm; }
    }
    __syncthreads();
}

// name_2k (D) from name_k (S).  Positions whose k-gram at p or at p + k occurs nowhere else are
// heads by construction and do not enter the table.  Also lists the participants of the bracket
// (k, 2k) in c.L: heads of their 2k-gram whose k-gram occurs elsewhere, with room for k+1 bytes
// (count in c.red[30]).  Returns "any match of 2k bytes".
__device__ inline int lz2_double(ChunkCtx &c, const uint16_t *S, uint16_t *D, int k)
{
    const int n = c.n, tid = threadIdx.x, lane = tid & 31;
    lz2_clear(c, LZ2_TSLOTS);
    volatile int *cnt = c.red + 30;
    if (tid == 0) *cnt = 0;
    __syncthreads();
    const int P = n - 2 * k + 1;
    int dummy = 0;
    for (int p = tid; p < n; p += AMBC_BLOCK) {
        uint32_t slot = 0xFFFFu;
        if (p < P) {
            const uint32_t a = S[p], b = S[p + k];
            if (a & b & LZ2_NS) {
                const uint32_t h = lz2_hash((a & 0xFFFu) | ((b & 0xFFFu) << 12), 0x7FFFFFFFu);
                slot = lz2_insert_pair(c, LZ2_TSLOTS - 1, h, S, a, b, p, k, &dummy);
            }
        }
        D[p] = (uint16_t)slot;
    }
    __syncthreads();
    uint16_t *plist = (uint16_t *)c.L;
    const int Pmax = n - k - 1;
    int nonhead = 0;
    for (int pb = 0; pb < n; pb += AMBC_BLOCK) {
        const int p = pb + tid;
        bool part = false;
        if (p < n) {
            const uint32_t slot = D[p];
            uint32_t nm = (uint32_t)p;
            if (slot != 0xFFFFu) nm = lz2_slot_name(c.T[slot]);
            D[p] = (uint16_t)nm;
            if ((nm & 0xFFFu) < (uint32_t)p) {
                c.mlen[p] = (uint8_t)(2 * k); c.mpos[p] = (uint16_t)(nm & 0xFFFu);
                nonhead++;
            } else part = p <= Pmax && (S[p] & LZ2_NS);
        }
        const uint32_t m = __ballot_sync(FULL_MASK, part);
        if (m) {
            int base = 0;
            if (lane == 0) base = atomicAdd((int *)cnt, __popc(m));
            base = __shfl_sync(FULL_MASK, base, 0);
            if (part) plist[base + __popc(m & ((1u << lane) - 1))] = (uint16_t)p;
        }
    }
    return __syncthreads_or(nonhead);
}

// ---- lengths k+1 .. 2k-1 --------------------------------------------------------------------
// every participant enters every length (np > LZ2_BIN_MAXP, and the fallback of the binary order)
__device__ inline bool lz2_refine_flat(ChunkCtx &c, const uint16_t *S, int k, int np, const uint16_t *plist, uint16_t *islot)
{
    const int n = c.n, tid = threadIdx.x;
    volatile int *ovf = c.red + 31;
    if (tid == 0) *ovf = 0;
    // pass = (group of nj consecutive lengths) x (one of R key partitions)
    int G = LZ2_PART_TARGET / np, R = 1;
    if (G < 1) { G = 1; while (R * LZ2_PART_TARGET < np) R <<= 1; }
    for (int j0 = 1; j0 < k; j0 += G) {
        const int nj = min(G, k - j0);
        for (int r = 0; r < R; r++) {
            lz2_clear(c, LZ2_RSLOTS);
            __syncthreads();
            int overflow = 0;
            for (int jj = 0; jj < nj; jj++) {
                const int j = j0 + jj;
                for (int pi = tid; pi < np; pi += AMBC_BLOCK) {
                    const int p = plist[pi];
                    uint32_t slot = 0xFFFFu;
                    if (p + k + j <= n) {
                        const uint32_t a = S[p], b = S[p + j];
                        if (b & LZ2_NS) {
                            const uint32_t h = lz2_hash((a & 0xFFFu) | ((b & 0xFFFu) << 12) | ((uint32_t)jj << 24), 0x7FFFFFFFu);
                            if (((h >> 7) & (uint32_t)(R - 1)) == (uint32_t)r)
                                slot = lz2_insert_pair(c, LZ2_RSLOTS - 1, h, S, a, b, p, j, &overflow);
                        }
                    }
                    islot[jj * np + pi] = (uint16_t)slot;
                }
            }
            if (overflow) *ovf = 1;
            __syncthreads();
            for (int pi = tid; pi < np; pi += AMBC_BLOCK) { // one thread owns all lengths of a participant
                const int p = plist[pi];
                for (int jj = nj - 1; jj >= 0; jj--) {       // longest first: a match implies the shorter ones
                    const uint32_t slot = islot[jj * np + pi];
                    if (slot == 0xFFFFu) continue;
                    const uint32_t nm = lz2_slot_pos(c.T[slot]);
                    if (nm < (uint32_t)p) {
                        const int L = k + j0 + jj;
                        if (L > (int)c.mlen[p]) { c.mlen[p] = (uint8_t)L; c.mpos[p] = (uint16_t)nm; }
                        break;
                    }
                }
            }
            __syncthreads();
            if (*ovf) return false;
        }
    }
    return true;
}

// Binary-search order with dense item lists.  An item = (node t << 12 | position): participant at
// node t of the current round.  Round 1's list is the participant list itself (t = 0); the resolve
// pass of a round appends the children items of the next round (left child 2t: the participant is a
// head at this length; right child 2t+1: the gram occurs elsewhere), so every pass runs over a dense
// list with one item per lane.  A participant matches at most once per round (a head at the common
// ancestor length cannot match above it), so mlen / mpos are written without atomics.
// Returns 0 = done, 1 = a list would overflow (caller rebuilds the participant list and runs the flat
// method).  Lists: three arrays of LZ2_LISTCAP items in c.L.
#ifndef LZ2_LOADINV
#define LZ2_LOADINV 4  // table slots per entry in the refinement rounds (1/4 load: measured best of 2..4)
#endif
#define LZ2_LISTCAP 5461
__device__ inline int lz2_refine_binary_dense(ChunkCtx &c, const uint16_t *S, int k, int np)
{
    const int n = c.n, tid = threadIdx.x, lane = tid & 31;
    uint16_t *A = (uint16_t *)c.L, *B = A + LZ2_LISTCAP, *islot = B + LZ2_LISTCAP;
    int E = np, dummy = 0, round = 0;
    for (int step = k >> 1; step >= 1; step >>= 1, round++) {
        // two alternating counters: the one of this round was last read two rounds ago
        volatile int *cntB = c.red + 28 + (round & 1);
        if (E == 0) return 0;
        // table of this round: the smallest power of two with load factor <= 1/2 (E < slot count always)
        const int tbits = min(13, max(10, 32 - __clz(LZ2_LOADINV * E - 1))); // smallest power of two >= LOADINV * E
        const uint32_t tmask = (1u << tbits) - 1u, wmask = (1u << (tbits + 18)) - 1u;
        lz2_clear(c, 1 << tbits);
        if (tid == 0) *cntB = 0;
        __syncthreads();
        for (int i = tid; i < E; i += AMBC_BLOCK) {
            const uint32_t item = A[i];
            const int p = item & 0xFFFu, t = item >> 12;
            const int j = (2 * t + 1) * step;
            uint32_t slot = 0xFFFEu; // 0xFFFE: unique by construction (head, no follower)
            if (p + k + j <= n) {
                const uint32_t a = S[p], b = S[p + j];
                if (b & LZ2_NS) {
                    const uint32_t h = lz2_hash((a & 0xFFFu) | ((b & 0xFFFu) << 12) | ((uint32_t)t << 24), wmask);
                    slot = lz2_insert_pair(c, tmask, h, S, a, b, p, j, &dummy);
                }
            }
            islot[i] = (uint16_t)slot;
        }
        __syncthreads();
        bool overflow = false;
        for (int ib = 0; ib < E; ib += AMBC_BLOCK) {
            const int i = ib + tid;
            bool left = false, right = false;
            uint32_t p = 0, t = 0;
            if (i < E) {
                const uint32_t item = A[i];
                p = item & 0xFFFu; t = item >> 12;
                const uint32_t slot = islot[i];
                if (slot == 0xFFFEu) left = true;
                else {
                    const uint32_t v = c.T[slot];
                    const uint32_t nm = lz2_slot_pos(v);
                    if (nm < p) {
                        // after a match a participant only visits longer lengths (it goes right), and a head
                        // at 2k held at most k before the bracket: the new length is always the longest so far
                        c.mlen[p] = (uint8_t)(k + (2 * (int)t + 1) * step);
                        c.mpos[p] = (uint16_t)nm;
                    } else left = true;      // head at this length: the lengths below remain
                    right = !(v & 1u);       // occurs elsewhere: the lengths above remain
                }
            }
            if (step > 1) {
                const uint32_t ml = __ballot_sync(FULL_MASK, left), mr = __ballot_sync(FULL_MASK, right);
                const int nl = __popc(ml), nr = __popc(mr);
                if (nl + nr) {
                    int base = 0;
                    if (lane == 0) base = atomicAdd((int *)cntB, nl + nr);
                    base = __shfl_sync(FULL_MASK, base, 0);
                    const uint32_t below = (1u << lane) - 1u;
                    if (base + nl + nr <= LZ2_LISTCAP) {
                        if (left) B[base + __popc(ml & below)] = (uint16_t)(((2u * t) << 12) | p);
                        if (right) B[base + nl + __popc(mr & below)] = (uint16_t)(((2u * t + 1u) << 12) | p);
                    } else overflow = true;
                }
            }
        }
        const int ov = __syncthreads_or(overflow);
        if (ov) return 1;
        E = *cntB;
        uint16_t *tmp = A; A = B; B = tmp;
    }
    return 0;
}

// S = name_k, D = name_2k.  Returns false on table overflow.
__device__ inline bool lz2_refine(ChunkCtx &c, const uint16_t *S, const uint16_t *D, int k)
{
    const int np = c.red[30]; // listed by lz2_double
    if (np == 0) return true;
    uint16_t *plist = (uint16_t *)c.L;
    if (k >= LZ2_BIN_MINK && np <= LZ2_LISTCAP) {
        if (lz2_refine_binary_dense(c, S, k, np) == 0) return true;
        // (rare) the item lists outgrew their memory: list the participants again, every length below
        const int n = c.n, tid = threadIdx.x, lane = tid & 31;
        volatile int *cnt = c.red + 30;
        __syncthreads();
        if (tid == 0) *cnt = 0;
        __syncthreads();
        for (int pb = 0; pb < n; pb += AMBC_BLOCK) {
            const int p = pb + tid;
            const bool part = p <= n - k - 1 && (D[p] & 0xFFFu) == (uint32_t)p && (S[p] & LZ2_NS);
            const uint32_t m = __ballot_sync(FULL_MASK, part);
            if (m) {
                int base = 0;
                if (lane == 0) base = atomicAdd((int *)cnt, __popc(m));
                base = __shfl_sync(FULL_MASK, base, 0);
                if (part) plist[base + __popc(m & ((1u << lane) - 1))] = (uint16_t)p;
            }
        }
        __syncthreads();
    }
    // flat method: plist 8 KiB | islot 16 KiB
    return lz2_refine_flat(c, S, k, c.red[30], plist, (uint16_t *)(c.L + 8192));
}

// mlen / mpos for every position of the chunk (c.mlen zeroed by the caller).  n <= LZ2_NMAX.
// Returns 0 = done, 1 = a table overflowed (run the bucket search).
__device__ inline int lz2_match_all(ChunkCtx &c)
{
    uint16_t *A = c.nameA, *B = c.nameB;
    if (c.n < 3) return 0;
    const int any4 = lz2_level4(c, A);
    lz2_level3(c, B);
    if (!any4) return 0;
    const int any8 = lz2_double(c, A, B, 4);
    if (!lz2_refine(c, A, B, 4)) return 1;
    if (!any8) return 0;
    const int any16 = lz2_double(c, B, A, 8);
    if (!lz2_refine(c, B, A, 8)) return 1;
    if (!any16) return 0;
    lz2_double(c, A, B, 16);
    const bool ok = lz2_refine(c, A, B, 16);
    return ok ? 0 : 1;
}
