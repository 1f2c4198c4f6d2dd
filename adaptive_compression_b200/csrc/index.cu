// index.cu -- GPU-side package index: the table ambc_index_host builds by walking the package chain
// on the host (adaptive_compressor.py:396-430, :444-445), built on the device instead.
//
// The chain is pointer chasing (pos += header + comp_len), but every package starts with the
// marker, so:
//   1. k_idx_scan   finds every occurrence of the marker bytes in the body (coalesced loads, matches
//                   into a shared-memory bitmap, ordered compaction) -> sorted candidate positions.
//                   The marker is NOT guaranteed absent from payloads (SURVEY.md D3), so candidates
//                   are a superset of the package starts;
//   2. k_idx_link   parses the header at every candidate and finds its successor (the candidate at
//                   pos + header + comp_len, by binary search), or why the walk would end there;
//   3. k_idx_jump   builds jump tables succ^(2^k); k_idx_end walks them from candidate 0 to the
//                   chain length, k_idx_chain lists the chain in order (binary lifting) -- only
//                   candidates reachable from position 0 are packages, exactly as in the serial walk;
//   4. scans of the nominal output sizes place every package (the walk stops once the output is
//                   complete, :444-445), raw packages are split into 64 KiB entries, and
//                   k_idx_emit writes the table.
// A marker mismatch the serial walk would hit is reported as AMBC_E_MARKER.
#include "ambc_internal.h"
#include "common.cuh"

#define IDX_TILE 16384   // body bytes per CTA in the marker scan
#define IDX_THREADS 256
#define IDX_RAW_PIECE 65536u
#define SC_TILE 2048     // elements per CTA in the device-wide scans

// ---- device-wide exclusive scan of uint64 (three small kernels) ----------------------------------
__global__ void __launch_bounds__(256) k_sc_tiles(const unsigned long long *__restrict__ v, uint64_t n, unsigned long long *tile)
{
    __shared__ unsigned long long red[8];
    const uint64_t base = (uint64_t)blockIdx.x * SC_TILE;
    unsigned long long s = 0;
    for (int k = threadIdx.x; k < SC_TILE; k += 256)
        if (base + k < n) s += v[base + k];
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(FULL_MASK, s, d);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int i = 0; i < 8; i++) t += red[i];
        tile[blockIdx.x] = t;
    }
}
__global__ void __launch_bounds__(1024) k_sc_top(unsigned long long *tile, uint64_t n_tiles, unsigned long long *total)
{
    __shared__ unsigned long long wsum[32];
    __shared__ unsigned long long carry_s;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid == 0) carry_s = 0;
    __syncthreads();
    for (uint64_t base = 0; base < n_tiles; base += 1024) {
        const uint64_t i = base + tid;
        unsigned long long v = i < n_tiles ? tile[i] : 0, inc = v;
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long t = __shfl_up_sync(FULL_MASK, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) wsum[w] = inc;
        __syncthreads();
        unsigned long long wbase = 0;
        for (int k = 0; k < w; k++) wbase += wsum[k];
        const unsigned long long carry = carry_s;
        if (i < n_tiles) tile[i] = carry + wbase + inc - v;
        __syncthreads();
        if (tid == 1023) carry_s = carry + wbase + inc;
        __syncthreads();
    }
    if (tid == 0) *total = carry_s;
}
__global__ void __launch_bounds__(256) k_sc_apply(const unsigned long long *__restrict__ v, uint64_t n,
                                                  const unsigned long long *__restrict__ tile, unsigned long long *out)
{
    __shared__ unsigned long long wsum[8];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const uint64_t base = (uint64_t)blockIdx.x * SC_TILE + (uint64_t)tid * 8;
    unsigned long long x[8], s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) { x[k] = base + k < n ? v[base + k] : 0; s += x[k]; }
    unsigned long long inc = s;
    for (int d = 1; d < 32; d <<= 1) {
        unsigned long long t = __shfl_up_sync(FULL_MASK, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    unsigned long long run = tile[blockIdx.x] + inc - s;
    for (int k = 0; k < w; k++) run += wsum[k];
#pragma unroll
    for (int k = 0; k < 8; k++) {
        if (base + k < n) out[base + k] = run;
        run += x[k];
    }
}
// out[i] = sum of v[0..i); *total = sum of all.  tile: >= ceil(n / SC_TILE) + 1 words of scratch.
static int dev_excl_scan(const unsigned long long *v, uint64_t n, unsigned long long *out, unsigned long long *tile,
                         unsigned long long *total, cudaStream_t s)
{
    const uint64_t nt = (n + SC_TILE - 1) / SC_TILE;
    if (n == 0) { CUDA_TRY(cudaMemsetAsync(total, 0, 8, s)); return AMBC_OK; }
    k_sc_tiles<<<(unsigned)nt, 256, 0, s>>>(v, n, tile);
    k_sc_top<<<1, 1024, 0, s>>>(tile, nt, total);
    k_sc_apply<<<(unsigned)nt, 256, 0, s>>>(v, n, tile, out);
    for (int i = 0; i < 3; i++) ambc_count_launch();
    CUDA_TRY(cudaGetLastError());
    return AMBC_OK;
}

// ---- 1. marker scan -------------------------------------------------------------------------------
// WRITE == false: tile_cnt[tile] = matches in the tile; WRITE == true: positions written in order at
// tile_base[tile].  A match at p needs p + mb <= len.
template <bool WRITE>
__global__ void __launch_bounds__(IDX_THREADS)
k_idx_scan(const uint8_t *__restrict__ body, uint64_t len, uint32_t marker_word, uint32_t mb,
           unsigned long long *tile_cnt, const unsigned long long *__restrict__ tile_base, unsigned long long *cand)
{
    __shared__ uint32_t bits[IDX_TILE / 32];
    __shared__ int wsum[IDX_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const uint64_t t0 = (uint64_t)blockIdx.x * IDX_TILE;
    for (int i = tid; i < IDX_TILE / 32; i += IDX_THREADS) bits[i] = 0;
    __syncthreads();
    const uint32_t kmask = mb >= 4 ? 0xFFFFFFFFu : ((1u << (8 * mb)) - 1u);
    if (((uintptr_t)body & 15) == 0 && t0 + IDX_TILE + 16 <= len) {
        // full tile, aligned: 16 bytes (+ one halo word) per thread and step, 16 windows each
        const uint4 *b4 = (const uint4 *)(body + t0);
        for (int j = 0; j < IDX_TILE / 16 / IDX_THREADS; j++) {
            const int v = j * IDX_THREADS + tid;
            const uint4 x = __ldg(b4 + v);
            const uint32_t halo = __ldg((const uint32_t *)(b4 + v + 1));
            const uint32_t w[5] = {x.x, x.y, x.z, x.w, halo};
            uint32_t m16 = 0;
#pragma unroll
            for (int b = 0; b < 16; b++) {
                const uint32_t win = __funnelshift_r(w[b >> 2], w[(b >> 2) + 1], (b & 3) * 8);
                if ((win & kmask) == marker_word) m16 |= 1u << b;
            }
            if (m16) atomicOr(&bits[v >> 1], m16 << ((v & 1) * 16));
        }
    } else {
        for (int j = 0; j < IDX_TILE / IDX_THREADS; j++) {
            const uint32_t q = (uint32_t)j * IDX_THREADS + tid; // coalesced: consecutive lanes, consecutive bytes
            const uint64_t p = t0 + q;
            if (p + mb <= len) {
                uint32_t v = 0;
                for (uint32_t k = 0; k < mb; k++) v |= (uint32_t)__ldg(body + p + k) << (8 * k);
                if ((v & kmask) == marker_word) atomicOr(&bits[q >> 5], 1u << (q & 31));
            }
        }
    }
    __syncthreads();
    // thread t owns words 2t, 2t+1 (64 consecutive positions)
    const uint32_t b0 = bits[2 * tid], b1 = bits[2 * tid + 1];
    const int mine = __popc(b0) + __popc(b1);
    int inc = mine;
    for (int d = 1; d < 32; d <<= 1) {
        int t = __shfl_up_sync(FULL_MASK, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    int base = inc - mine, tot = 0;
    for (int k = 0; k < IDX_THREADS / 32; k++) { if (k < w) base += wsum[k]; tot += wsum[k]; }
    if (!WRITE) {
        if (tid == 0) tile_cnt[blockIdx.x] = (unsigned long long)tot;
    } else {
        unsigned long long *dst = cand + tile_base[blockIdx.x] + base;
        uint32_t x = b0;
        while (x) { const int b = __ffs(x) - 1; x &= x - 1; *dst++ = t0 + 64ull * tid + b; }
        x = b1;
        while (x) { const int b = __ffs(x) - 1; x &= x - 1; *dst++ = t0 + 64ull * tid + 32 + b; }
    }
}

// ---- 2. headers and successors ----------------------------------------------------------------------
struct IdxRec {
    uint32_t orig, comp;
    uint8_t type, kind; // kind: 0 package, 1 END, 2 header cut off, 3 payload cut off
    uint16_t pad;
};
#define IDX_STOP(M) ((uint32_t)(M))      // the walk ends here without error
#define IDX_ERR(M) ((uint32_t)(M) + 1u)  // the walk raises "Marker mismatch" at the next position

__global__ void __launch_bounds__(256)
k_idx_link(const uint8_t *__restrict__ body, uint64_t len, uint32_t mb, const unsigned long long *__restrict__ cand,
           uint32_t M, IdxRec *rec, uint32_t *succ)
{
    const uint32_t i = blockIdx.x * 256 + threadIdx.x;
    if (i >= M + 2) return;
    if (i >= M) { succ[i] = i; return; } // absorbing
    const uint64_t hdr = mb + 14, pos = cand[i];
    IdxRec r;
    r.orig = r.comp = 0; r.type = 0; r.kind = 0; r.pad = 0;
    uint32_t sx = IDX_STOP(M);
    if (pos + hdr > len) r.kind = 2;                                    // :400-403
    else {
        r.type = body[pos + mb];
        uint32_t o = 0, c = 0;
        for (int k = 0; k < 4; k++) { o |= (uint32_t)body[pos + mb + 6 + k] << (8 * k); c |= (uint32_t)body[pos + mb + 10 + k] << (8 * k); }
        r.orig = o; r.comp = c;
        const uint64_t nxt = pos + hdr + c;
        if (r.type == 0) r.kind = 1;                                    // :422-424
        else if (nxt > len) r.kind = 3;                                 // :425-427
        else if (nxt + hdr > len) sx = IDX_STOP(M);                     // the next iteration stops at :400-403 (or pos == len)
        else {
            uint32_t lo = i + 1, hi = M; // candidates are sorted; nxt > pos
            while (lo < hi) { const uint32_t mid = lo + (hi - lo) / 2; if (cand[mid] < nxt) lo = mid + 1; else hi = mid; }
            sx = (lo < M && cand[lo] == nxt) ? lo : IDX_ERR(M);         // :405-407
        }
    }
    rec[i] = r;
    succ[i] = sx;
}

// ---- 3. jump tables, chain ----------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_idx_jump(const uint32_t *__restrict__ prev, uint32_t *next, uint32_t n)
{
    const uint32_t i = blockIdx.x * 256 + threadIdx.x;
    if (i < n) next[i] = prev[prev[i]];
}
// info[0] = chain length (nodes visited from candidate 0), info[1] = 1 when the walk ends in a marker mismatch
__global__ void k_idx_end(const uint32_t *__restrict__ J, uint32_t n, int K, uint32_t M, unsigned long long *info)
{
    if (threadIdx.x || blockIdx.x) return;
    uint32_t node = 0;
    unsigned long long steps = 0;
    for (int k = K - 1; k >= 0; k--) {
        const uint32_t nx = J[(uint64_t)k * n + node];
        if (nx < M) { node = nx; steps += 1ull << k; }
    }
    info[0] = steps + 1;
    info[1] = J[node] == IDX_ERR(M) ? 1 : 0;
}
__global__ void __launch_bounds__(256)
k_idx_chain(const uint32_t *__restrict__ J, uint32_t n, int K, uint64_t chain_len, uint32_t *chain)
{
    const uint64_t r = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (r >= chain_len) return;
    uint32_t node = 0;
    for (int k = 0; k < K; k++)
        if ((r >> k) & 1) node = J[(uint64_t)k * n + node];
    chain[r] = node;
}

// ---- 4. placement and table ------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t idx_nominal(uint32_t type, bool known, uint32_t comp, uint32_t orig)
{
    if (!known) return comp;                       // copied through (:432-435)
    switch (type) {
    case 255: return orig;                         // pad / truncate (compression_methods.py:703-713)
    case 4: return comp == 0 ? 0 : (comp < orig ? comp : orig); // :621-638
    default: return comp == 0 ? 0 : orig;          // `if not data: return b''`
    }
}
__device__ __forceinline__ bool idx_known(uint32_t type, uint32_t known_mask)
{
    return type == 255 || (type < 32 && ((known_mask >> type) & 1u));
}
__global__ void __launch_bounds__(256)
k_idx_nominal(const IdxRec *__restrict__ rec, const uint32_t *__restrict__ chain, uint64_t chain_len, uint32_t known_mask,
              unsigned long long *nominal)
{
    const uint64_t r = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (r >= chain_len) return;
    const IdxRec x = rec[chain[r]];
    nominal[r] = x.kind == 0 ? idx_nominal(x.type, idx_known(x.type, known_mask), x.comp, x.orig) : 0;
}
// cut = first chain rank after which the walk stops because the output is complete (:444-445)
__global__ void __launch_bounds__(256)
k_idx_cut(const unsigned long long *__restrict__ nominal, const unsigned long long *__restrict__ obefore, uint64_t chain_len,
          uint64_t orig_size, unsigned long long *cut)
{
    const uint64_t r = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (r >= chain_len) return;
    if (obefore[r] + nominal[r] >= orig_size) atomicMin(cut, (unsigned long long)r);
}
__global__ void __launch_bounds__(256)
k_idx_count(const IdxRec *__restrict__ rec, const uint32_t *__restrict__ chain, const unsigned long long *__restrict__ nominal,
            const unsigned long long *__restrict__ obefore, uint64_t chain_len, uint64_t orig_size, uint32_t known_mask,
            const unsigned long long *__restrict__ cut, unsigned long long *ecount)
{
    const uint64_t r = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (r >= chain_len) return;
    unsigned long long e = 0;
    const IdxRec x = rec[chain[r]];
    if (r <= *cut && x.kind == 0) {
        const uint64_t o = obefore[r], room = orig_size > o ? orig_size - o : 0;
        const uint64_t emit = nominal[r] < room ? nominal[r] : room;
        if (emit) e = (!idx_known(x.type, known_mask) || x.type == 255) ? (emit + IDX_RAW_PIECE - 1) / IDX_RAW_PIECE : 1;
    }
    ecount[r] = e;
}
__global__ void __launch_bounds__(256)
k_idx_emit(const IdxRec *__restrict__ rec, const uint32_t *__restrict__ chain, const unsigned long long *__restrict__ cand,
           const unsigned long long *__restrict__ nominal, const unsigned long long *__restrict__ obefore,
           const unsigned long long *__restrict__ ecount, const unsigned long long *__restrict__ ebase, uint64_t chain_len,
           uint64_t orig_size, uint32_t known_mask, uint32_t mb, ambc_pkg *table, uint64_t table_cap)
{
    const uint64_t r = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (r >= chain_len || ecount[r] == 0) return;
    const IdxRec x = rec[chain[r]];
    const uint64_t pos = cand[chain[r]] + mb + 14; // payload offset
    const uint64_t o = obefore[r], room = orig_size - o;
    const uint64_t emit = nominal[r] < room ? nominal[r] : room;
    uint64_t at = ebase[r];
    if (!idx_known(x.type, known_mask) || x.type == 255) {
        for (uint64_t done = 0; done < emit; done += IDX_RAW_PIECE, at++) {
            if (at >= table_cap) return;
            const uint64_t piece = emit - done < IDX_RAW_PIECE ? emit - done : IDX_RAW_PIECE;
            const uint64_t have = x.comp > done ? x.comp - done : 0;
            ambc_pkg e;
            e.src_off = pos + done; e.dst_off = o + done;
            e.comp_len = (uint32_t)(have < piece ? have : piece);
            e.orig_len = (uint32_t)piece; e.type = 255; e.out_len = (uint32_t)piece;
            table[at] = e;
        }
    } else if (at < table_cap) {
        ambc_pkg e;
        e.src_off = pos; e.dst_off = o; e.comp_len = x.comp; e.orig_len = x.orig; e.type = x.type; e.out_len = (uint32_t)emit;
        table[at] = e;
    }
}

// ---- host side ------------------------------------------------------------------------------------------------
struct IdxBuf {
    void *p = nullptr;
    uint64_t cap = 0;
    int ensure(uint64_t bytes)
    {
        if (bytes <= cap) return AMBC_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        const uint64_t want = bytes + bytes / 4 + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { p = nullptr; return ambc_fail(AMBC_E_CUDA, "cudaMalloc(%llu): %s", (unsigned long long)want, cudaGetErrorString(e)); }
        cap = want;
        return AMBC_OK;
    }
};
static IdxBuf g_idx_a[16], g_idx_b[16];

extern "C" int ambc_index_dev(const void *body_dev, uint64_t body_len, const uint8_t *marker, uint32_t mb, uint64_t orig_size,
                              uint32_t known_mask, ambc_pkg *table_dev, uint64_t table_cap, uint64_t *n_entries,
                              uint64_t *out_bytes, void *stream_)
{
    cudaStream_t s = (cudaStream_t)stream_;
    if (!marker || mb < 1 || mb > 4 || (body_len && !body_dev)) return ambc_fail(AMBC_E_ARG, "ambc_index_dev: bad argument");
    if (n_entries) *n_entries = 0;
    if (out_bytes) *out_bytes = 0;
    const uint64_t hdr = mb + 14;
    if (body_len < hdr) return AMBC_OK; // the walk stops before the first header (:400-403)
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 16) return ambc_fail(AMBC_E_ARG, "device index out of range");
    uint32_t marker_word = 0;
    for (uint32_t k = 0; k < mb; k++) marker_word |= (uint32_t)marker[k] << (8 * k);
    const uint8_t *body = (const uint8_t *)body_dev;

    // 1. candidates
    const uint64_t n_tiles = (body_len + IDX_TILE - 1) / IDX_TILE;
    IdxBuf &A = g_idx_a[dev], &B = g_idx_b[dev];
    int rc = A.ensure((n_tiles + 2) * 8 * 2 + ((n_tiles + SC_TILE) / SC_TILE + 2) * 8 + 64);
    if (rc) return rc;
    unsigned long long *tile_cnt = (unsigned long long *)A.p, *tile_base = tile_cnt + n_tiles + 1;
    unsigned long long *sc_tile = tile_base + n_tiles + 1, *d_total = sc_tile + (n_tiles + SC_TILE) / SC_TILE + 1;
    k_idx_scan<false><<<(unsigned)n_tiles, IDX_THREADS, 0, s>>>(body, body_len, marker_word, mb, tile_cnt, nullptr, nullptr);
    ambc_count_launch();
    if ((rc = dev_excl_scan(tile_cnt, n_tiles, tile_base, sc_tile, d_total, s))) return rc;
    unsigned long long h_total = 0;
    CUDA_TRY(cudaMemcpyAsync(&h_total, d_total, 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    const uint64_t M64 = h_total;
    if (M64 == 0) return ambc_fail(AMBC_E_MARKER, "Marker mismatch in chunk header."); // position 0 is not a marker
    if (M64 > 0x7FFFFFF0ull) return ambc_fail(AMBC_E_CAPACITY, "ambc_index_dev: too many marker occurrences");
    const uint32_t M = (uint32_t)M64, n = M + 2;
    int K = 1;
    while ((1ull << K) <= M) K++;
    // layout of B: cand | rec | J[K][n] | chain | nominal | obefore | ecount | ebase | scan tiles | info
    const uint64_t sc_tiles = (M64 + SC_TILE) / SC_TILE + 2;
    uint64_t off = 0;
    auto take = [&](uint64_t bytes) { uint64_t r = off; off += (bytes + 255) & ~255ull; return r; };
    const uint64_t o_cand = take(M64 * 8), o_rec = take(M64 * sizeof(IdxRec)), o_J = take((uint64_t)K * n * 4), o_chain = take(M64 * 4),
                   o_nom = take(M64 * 8), o_ob = take(M64 * 8), o_ec = take(M64 * 8), o_eb = take(M64 * 8), o_sct = take(sc_tiles * 8),
                   o_info = take(64);
    if ((rc = B.ensure(off))) return rc;
    uint8_t *W = (uint8_t *)B.p;
    unsigned long long *cand = (unsigned long long *)(W + o_cand);
    IdxRec *rec = (IdxRec *)(W + o_rec);
    uint32_t *J = (uint32_t *)(W + o_J), *chain = (uint32_t *)(W + o_chain);
    unsigned long long *nominal = (unsigned long long *)(W + o_nom), *obefore = (unsigned long long *)(W + o_ob);
    unsigned long long *ecount = (unsigned long long *)(W + o_ec), *ebase = (unsigned long long *)(W + o_eb);
    unsigned long long *sct = (unsigned long long *)(W + o_sct), *info = (unsigned long long *)(W + o_info);
    k_idx_scan<true><<<(unsigned)n_tiles, IDX_THREADS, 0, s>>>(body, body_len, marker_word, mb, nullptr, tile_base, cand);
    ambc_count_launch();
    unsigned long long first = 1;
    CUDA_TRY(cudaMemcpyAsync(&first, cand, 8, cudaMemcpyDeviceToHost, s));

    // 2. + 3. links, jump tables, chain
    k_idx_link<<<(n + 255) / 256, 256, 0, s>>>(body, body_len, mb, cand, M, rec, J);
    ambc_count_launch();
    for (int k = 1; k < K; k++) {
        k_idx_jump<<<(n + 255) / 256, 256, 0, s>>>(J + (uint64_t)(k - 1) * n, J + (uint64_t)k * n, n);
        ambc_count_launch();
    }
    k_idx_end<<<1, 1, 0, s>>>(J, n, K, M, info);
    ambc_count_launch();
    unsigned long long h_info[4] = {0, 0, 0, 0};
    CUDA_TRY(cudaMemcpyAsync(h_info, info, 16, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    if (first != 0) return ambc_fail(AMBC_E_MARKER, "Marker mismatch in chunk header."); // position 0 is not a marker
    const uint64_t chain_len = h_info[0];
    const bool ends_in_mismatch = h_info[1] != 0;
    const unsigned cgrid = (unsigned)((chain_len + 255) / 256);
    k_idx_chain<<<cgrid, 256, 0, s>>>(J, n, K, chain_len, chain);
    ambc_count_launch();

    // 4. placement
    k_idx_nominal<<<cgrid, 256, 0, s>>>(rec, chain, chain_len, known_mask, nominal);
    ambc_count_launch();
    if ((rc = dev_excl_scan(nominal, chain_len, obefore, sct, info + 2, s))) return rc;
    const unsigned long long none = ~0ull;
    CUDA_TRY(cudaMemcpyAsync(info + 3, &none, 8, cudaMemcpyHostToDevice, s));
    k_idx_cut<<<cgrid, 256, 0, s>>>(nominal, obefore, chain_len, orig_size, info + 3);
    k_idx_count<<<cgrid, 256, 0, s>>>(rec, chain, nominal, obefore, chain_len, orig_size, known_mask, info + 3, ecount);
    ambc_count_launch(); ambc_count_launch();
    if ((rc = dev_excl_scan(ecount, chain_len, ebase, sct, info + 4, s))) return rc;
    unsigned long long h_res[3] = {0, 0, 0}; // total nominal, cut, entries
    CUDA_TRY(cudaMemcpyAsync(h_res, info + 2, 24, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    const uint64_t cut = h_res[1], ne = h_res[2];
    if (ends_in_mismatch && cut == ~0ull) return ambc_fail(AMBC_E_MARKER, "Marker mismatch in chunk header.");
    // bytes the walk produced: everything up to and including the cut package
    uint64_t produced = h_res[0];
    if (cut != ~0ull) {
        unsigned long long ob = 0, nm = 0;
        CUDA_TRY(cudaMemcpyAsync(&ob, obefore + cut, 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(&nm, nominal + cut, 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        produced = ob + nm;
    }
    if (n_entries) *n_entries = ne;
    if (out_bytes) *out_bytes = produced < orig_size ? produced : orig_size;
    if (table_dev) {
        if (ne > table_cap) return ambc_fail(AMBC_E_CAPACITY, "ambc_index_dev: table too small (%llu entries)", (unsigned long long)ne);
        k_idx_emit<<<cgrid, 256, 0, s>>>(rec, chain, cand, nominal, obefore, ecount, ebase, chain_len, orig_size, known_mask, mb,
                                        table_dev, table_cap);
        ambc_count_launch();
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaStreamSynchronize(s));
    }
    return AMBC_OK;
}

// ==== range-local index (ambc_range_*): one rank's byte range [lo, hi) of the body ============================
// The walk above, split across ranks.  Candidates are the marker occurrences that start in [lo, hi); nodes
// M (stop) and M + 1 (marker mismatch) are those of k_idx_link, node M + 2 is an exit: the successor lies at
// or beyond hi, in a later range.  Next to J[k] = succ^(2^k) the range keeps S[k][i] = output bytes of the
// 2^k packages from node i on (the k_idx_nominal rule), so that one lifting pass from any candidate finds
// where the chain leaves the range or where the walk ends (the stop rule :444-445 included), and how many
// output bytes lie on the way.  The fold (k_rng_fold) runs that pass from the state the previous range
// handed on; ambc_range_table lists the chain from there and places every entry with global output offsets.
#define RNG_EXIT(M) ((uint32_t)(M) + 2u)

struct RngGeo { // body positions are global
    uint64_t lo, hi, body_len, orig_size;
    uint32_t mb, known_mask;
};
struct RngShare { uint64_t a, b; };

__host__ __device__ __forceinline__ uint64_t rng_min(uint64_t x, uint64_t y) { return x < y ? x : y; }
__host__ __device__ __forceinline__ uint64_t rng_nominal(uint32_t type, uint32_t known_mask, uint32_t comp, uint32_t orig)
{
    const bool known = type == 255 || (type < 32 && ((known_mask >> type) & 1u));
    if (!known) return comp;
    if (type == 255) return orig;
    if (type == 4) return comp == 0 ? 0 : (comp < orig ? comp : orig);
    return comp == 0 ? 0 : orig;
}
__host__ __device__ __forceinline__ bool rng_copied(uint32_t type, uint32_t known_mask)
{
    return type == 255 || !(type < 32 && ((known_mask >> type) & 1u));
}
// bytes the walk emits for a package with `nominal` output bytes at output offset o
__host__ __device__ __forceinline__ uint64_t rng_emit(uint64_t nominal, uint64_t o, uint64_t orig_size)
{
    return rng_min(nominal, orig_size > o ? orig_size - o : 0);
}
// the output bytes [a, b) of a copied-through package (payload at body position pay) that the range [lo, hi)
// owns: the payload bytes it holds, plus the zero pad when it holds the payload's last byte; the range that
// holds the header owns everything before its end.
__host__ __device__ __forceinline__ RngShare rng_share(uint64_t pay, uint64_t comp, uint64_t emit, uint64_t lo, uint64_t hi,
                                                       bool header_here)
{
    RngShare s;
    s.a = s.b = 0;
    if (!header_here && pay + comp <= lo) return s; // the payload ended in an earlier range
    s.a = header_here ? 0 : rng_min(lo > pay ? lo - pay : 0, emit);
    s.b = pay + comp <= hi ? emit : rng_min(hi > pay ? hi - pay : 0, emit);
    if (s.b < s.a) s.b = s.a;
    return s;
}
// first output byte owned by the range starting at body position lo, given the state handed to it
static uint64_t rng_out_offset(const ambc_range_state &s, uint64_t lo, uint64_t orig_size, uint32_t mb, uint32_t known_mask)
{
    if (s.pkg_pos != AMBC_RANGE_NO_PKG && rng_copied(s.pkg_type, known_mask)) {
        const uint64_t pay = s.pkg_pos + mb + 14;
        if (pay + s.pkg_comp > lo) {
            const uint64_t emit = rng_emit(rng_nominal(s.pkg_type, known_mask, s.pkg_comp, s.pkg_orig), s.pkg_out, orig_size);
            return rng_min(s.pkg_out + rng_share(pay, s.pkg_comp, emit, lo, ~0ull, false).a, orig_size);
        }
    }
    return rng_min(s.out_before, orig_size);
}

__global__ void __launch_bounds__(256)
k_rng_link(const uint8_t *__restrict__ buf, RngGeo g, const unsigned long long *__restrict__ cand, uint32_t M, IdxRec *rec,
           uint32_t *succ, unsigned long long *sum)
{
    const uint32_t i = blockIdx.x * 256 + threadIdx.x;
    if (i >= M + 3) return;
    if (i >= M) { succ[i] = i; sum[i] = 0; return; } // absorbing
    const uint64_t hdr = g.mb + 14, p = cand[i], pos = g.lo + p;
    IdxRec r;
    r.orig = r.comp = 0; r.type = 0; r.kind = 0; r.pad = 0;
    uint32_t sx = IDX_STOP(M);
    if (pos + hdr > g.body_len) r.kind = 2;                           // :400-403
    else {
        r.type = buf[p + g.mb];
        uint32_t o = 0, c = 0;
        for (int k = 0; k < 4; k++) { o |= (uint32_t)buf[p + g.mb + 6 + k] << (8 * k); c |= (uint32_t)buf[p + g.mb + 10 + k] << (8 * k); }
        r.orig = o; r.comp = c;
        const uint64_t nxt = pos + hdr + c;
        if (r.type == 0) r.kind = 1;                                    // :422-424
        else if (nxt > g.body_len) r.kind = 3;                          // :425-427
        else if (nxt + hdr > g.body_len) sx = IDX_STOP(M);              // the next iteration stops at :400-403
        else if (nxt >= g.hi) sx = RNG_EXIT(M);                         // a later range continues
        else {
            const uint64_t want = nxt - g.lo;
            uint32_t lo = i + 1, hi = M;
            while (lo < hi) { const uint32_t mid = lo + (hi - lo) / 2; if (cand[mid] < want) lo = mid + 1; else hi = mid; }
            sx = (lo < M && cand[lo] == want) ? lo : IDX_ERR(M);        // :405-407
        }
    }
    rec[i] = r;
    succ[i] = sx;
    sum[i] = r.kind == 0 ? rng_nominal(r.type, g.known_mask, r.comp, r.orig) : 0;
}
__global__ void __launch_bounds__(256)
k_rng_jump(const uint32_t *__restrict__ pj, const unsigned long long *__restrict__ ps, uint32_t *nj, unsigned long long *ns, uint32_t n)
{
    const uint32_t i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const uint32_t a = pj[i];
    nj[i] = pj[a];
    ns[i] = ps[i] + ps[a];
}
// one fold step.  walk[0] = chain length in this range from the entry (0: the walk does not pass here),
// walk[1] = entry node, walk[2] = last node, walk[3] = output offset of the last node
__global__ void k_rng_fold(const unsigned long long *__restrict__ cand, const IdxRec *__restrict__ rec, const uint32_t *__restrict__ J,
                           const unsigned long long *__restrict__ S, uint32_t n, int K, uint32_t M, RngGeo g,
                           const ambc_range_state *in, ambc_range_state *out, unsigned long long *walk)
{
    if (threadIdx.x || blockIdx.x) return;
    ambc_range_state s = *in;
    walk[0] = 0; walk[1] = walk[2] = M; walk[3] = 0;
    if (s.status != AMBC_RANGE_RUNNING || s.next_pos < g.lo || s.next_pos >= g.hi) { *out = s; return; }
    const uint64_t hdr = g.mb + 14, x = s.next_pos - g.lo;
    uint32_t a = 0, b = M;
    while (a < b) { const uint32_t mid = a + (b - a) / 2; if (cand[mid] < x) a = mid + 1; else b = mid; }
    s.pkg_pos = AMBC_RANGE_NO_PKG;
    if (a == M || cand[a] != x) { // no marker here: the walk stops (:400-403) or raises (:405-407)
        s.status = s.next_pos + hdr > g.body_len ? AMBC_RANGE_TRUNCATED : AMBC_RANGE_MARKER;
        *out = s;
        return;
    }
    uint32_t node = a;
    unsigned long long acc = s.out_before, steps = 0;
    for (int k = K - 1; k >= 0; k--) {
        const uint64_t at = (uint64_t)k * n + node;
        if (J[at] < M && acc + S[at] < g.orig_size) { acc += S[at]; node = J[at]; steps += 1ull << k; }
    }
    walk[0] = steps + 1; walk[1] = a; walk[2] = node; walk[3] = acc;
    const IdxRec r = rec[node];
    s.out_before = acc + S[node];
    if (r.kind == 1) s.status = AMBC_RANGE_END;
    else if (r.kind != 0) s.status = AMBC_RANGE_TRUNCATED;
    else {
        const uint64_t pos = g.lo + cand[node], end = pos + hdr + r.comp;
        if (end > g.hi) { s.pkg_pos = pos; s.pkg_out = acc; s.pkg_type = r.type; s.pkg_orig = r.orig; s.pkg_comp = r.comp; }
        const uint32_t sx = J[node];
        if (s.out_before >= g.orig_size) s.status = AMBC_RANGE_COMPLETE; // :444-445 before the next header is read
        else if (sx == IDX_STOP(M)) s.status = AMBC_RANGE_TRUNCATED;
        else if (sx == IDX_ERR(M)) s.status = AMBC_RANGE_MARKER;
        else s.next_pos = end;                                            // exit: a later range holds it
    }
    *out = s;
}
__global__ void __launch_bounds__(256)
k_rng_chain(const uint32_t *__restrict__ J, uint32_t n, int K, uint32_t entry, uint64_t chain_len, uint32_t *chain)
{
    const uint64_t r = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (r >= chain_len) return;
    uint32_t node = entry;
    for (int k = 0; k < K; k++)
        if ((r >> k) & 1) node = J[(uint64_t)k * n + node];
    chain[r] = node;
}
__device__ __forceinline__ void rng_put_pieces(ambc_pkg *table, uint64_t at, uint64_t pay, uint32_t comp, RngShare sh, uint64_t o,
                                               uint64_t lo, uint64_t out_lo)
{
    for (uint64_t done = sh.a; done < sh.b; done += IDX_RAW_PIECE, at++) {
        const uint64_t piece = rng_min(sh.b - done, IDX_RAW_PIECE), have = comp > done ? comp - done : 0;
        ambc_pkg e;
        e.src_off = pay - lo + done; e.dst_off = o + done - out_lo;
        e.comp_len = (uint32_t)rng_min(have, piece);
        e.orig_len = (uint32_t)piece; e.type = 255; e.out_len = (uint32_t)piece;
        table[at] = e;
    }
}
// WRITE == false: ecount[r] = entries of chain node r; WRITE == true: write them at base + ebase[r]
template <bool WRITE>
__global__ void __launch_bounds__(256)
k_rng_entries(const IdxRec *__restrict__ rec, const uint32_t *__restrict__ chain, const unsigned long long *__restrict__ cand,
              const unsigned long long *__restrict__ nominal, const unsigned long long *__restrict__ obefore, uint64_t chain_len,
              uint64_t out0, RngGeo g, unsigned long long *ecount, const unsigned long long *__restrict__ ebase, uint64_t base,
              uint64_t out_lo, ambc_pkg *table)
{
    const uint64_t r = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (r >= chain_len) return;
    const IdxRec x = rec[chain[r]];
    const uint64_t o = out0 + obefore[r], emit = x.kind == 0 ? rng_emit(nominal[r], o, g.orig_size) : 0;
    const uint64_t pay = g.lo + cand[chain[r]] + g.mb + 14;
    const bool copied = rng_copied(x.type, g.known_mask);
    const RngShare sh = rng_share(pay, x.comp, emit, g.lo, g.hi, true);
    if (!WRITE) {
        ecount[r] = emit == 0 ? 0 : copied ? (sh.b - sh.a + IDX_RAW_PIECE - 1) / IDX_RAW_PIECE : 1;
        return;
    }
    if (emit == 0) return;
    if (copied) {
        rng_put_pieces(table, base + ebase[r], pay, x.comp, sh, o, g.lo, out_lo);
    } else {
        ambc_pkg e;
        e.src_off = pay - g.lo; e.dst_off = o - out_lo; e.comp_len = x.comp; e.orig_len = x.orig; e.type = x.type;
        e.out_len = (uint32_t)emit;
        table[base + ebase[r]] = e;
    }
}
// the pieces of a copied-through package whose header lies in an earlier range
__global__ void __launch_bounds__(256)
k_rng_inbound(uint64_t pay, uint32_t comp, RngShare sh, uint64_t o, uint64_t lo, uint64_t out_lo, ambc_pkg *table)
{
    const uint64_t j = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    const uint64_t a = sh.a + j * IDX_RAW_PIECE;
    if (a >= sh.b) return;
    RngShare one;
    one.a = a; one.b = rng_min(sh.b, a + IDX_RAW_PIECE);
    rng_put_pieces(table, j, pay, comp, one, o, lo, out_lo);
}

struct RngLayout {
    uint64_t tile_cnt, tile_base, sc, total, cand, rec, J, S, chain, nom, ob, ec, eb, sct, info, bytes;
    uint32_t n;
    int K;
};
static RngLayout rng_layout(uint64_t range_len, uint64_t M)
{
    RngLayout l;
    const uint64_t n_tiles = (range_len + 3 + IDX_TILE - 1) / IDX_TILE; // the scan covers at most range_len + 3 bytes
    l.n = (uint32_t)(M + 3);
    l.K = 1;
    while ((1ull << l.K) <= M) l.K++;
    uint64_t off = 0;
    auto take = [&](uint64_t bytes) { uint64_t r = off; off += (bytes + 255) & ~255ull; return r; };
    l.tile_cnt = take((n_tiles + 1) * 8); l.tile_base = take((n_tiles + 1) * 8);
    l.sc = take(((n_tiles + SC_TILE) / SC_TILE + 1) * 8); l.total = take(8);
    l.cand = take(M * 8); l.rec = take(M * sizeof(IdxRec)); l.J = take((uint64_t)l.K * l.n * 4); l.S = take((uint64_t)l.K * l.n * 8);
    l.chain = take(M * 4); l.nom = take(M * 8); l.ob = take(M * 8); l.ec = take(M * 8); l.eb = take(M * 8);
    l.sct = take(((M + SC_TILE) / SC_TILE + 2) * 8); l.info = take(256);
    l.bytes = off;
    return l;
}
// info area: [0, 48) state in, [64, 112) state out, [128, 160) walk, [160, 192) scan totals
#define RNG_IN 0
#define RNG_OUT 64
#define RNG_WALK 128
#define RNG_TOT 160

extern "C" uint64_t ambc_range_workspace_bytes(uint64_t range_len, uint64_t n_cand)
{
    return rng_layout(range_len, n_cand).bytes;
}

extern "C" uint64_t ambc_range_out_offset(const ambc_range_state *s, uint64_t lo, uint64_t orig_size, uint32_t mb,
                                          uint32_t known_mask)
{
    return s ? rng_out_offset(*s, lo, orig_size, mb, known_mask) : 0;
}

static RngGeo rng_geo(const ambc_range *r)
{
    RngGeo g;
    g.lo = r->lo; g.hi = r->hi; g.body_len = r->body_len; g.orig_size = r->orig_size; g.mb = r->marker_bytes;
    g.known_mask = r->known_mask;
    return g;
}

extern "C" int ambc_range_index(const void *buf_dev, uint64_t buf_len, uint64_t lo, uint64_t hi, uint64_t body_len,
                                const uint8_t *marker, uint32_t mb, uint64_t orig_size, uint32_t known_mask, void *work_dev,
                                uint64_t work_bytes, ambc_range *r, void *stream_)
{
    cudaStream_t s = (cudaStream_t)stream_;
    if (!r || !marker || mb < 1 || mb > 4 || lo > hi || hi > body_len || (buf_len && !buf_dev))
        return ambc_fail(AMBC_E_ARG, "ambc_range_index: bad argument");
    const uint64_t halo_end = rng_min(hi + mb + 13, body_len);
    if (lo + buf_len < halo_end) return ambc_fail(AMBC_E_ARG, "ambc_range_index: buffer ends before the header halo");
    r->lo = lo; r->hi = hi; r->body_len = body_len; r->orig_size = orig_size; r->n_cand = 0;
    r->work_dev = work_dev; r->marker_bytes = mb; r->known_mask = known_mask; r->levels = 1; r->reserved = 0;
    const uint64_t R = hi - lo;
    RngLayout l = rng_layout(R, 0);
    r->work_bytes = l.bytes;
    if (!work_dev || work_bytes < l.bytes) return ambc_fail(AMBC_E_CAPACITY, "ambc_range_index: workspace too small");
    uint32_t marker_word = 0;
    for (uint32_t k = 0; k < mb; k++) marker_word |= (uint32_t)marker[k] << (8 * k);
    const uint8_t *buf = (const uint8_t *)buf_dev;
    uint8_t *W = (uint8_t *)work_dev;
    // candidates: marker occurrences that start in [lo, hi)
    const uint64_t scan_len = R ? rng_min(buf_len, R + mb - 1) : 0, n_tiles = (scan_len + IDX_TILE - 1) / IDX_TILE;
    unsigned long long *tile_cnt = (unsigned long long *)(W + l.tile_cnt), *tile_base = (unsigned long long *)(W + l.tile_base);
    uint64_t M64 = 0;
    int rc;
    if (n_tiles) {
        k_idx_scan<false><<<(unsigned)n_tiles, IDX_THREADS, 0, s>>>(buf, scan_len, marker_word, mb, tile_cnt, nullptr, nullptr);
        ambc_count_launch();
        unsigned long long *d_total = (unsigned long long *)(W + l.total);
        if ((rc = dev_excl_scan(tile_cnt, n_tiles, tile_base, (unsigned long long *)(W + l.sc), d_total, s))) return rc;
        unsigned long long h_total = 0;
        CUDA_TRY(cudaMemcpyAsync(&h_total, d_total, 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        M64 = h_total;
    }
    if (M64 > 0x7FFFFFF0ull) return ambc_fail(AMBC_E_CAPACITY, "ambc_range_index: too many marker occurrences");
    l = rng_layout(R, M64);
    r->n_cand = M64;
    r->work_bytes = l.bytes;
    r->levels = (uint32_t)l.K;
    if (work_bytes < l.bytes) return ambc_fail(AMBC_E_CAPACITY, "ambc_range_index: workspace too small (%llu bytes)", (unsigned long long)l.bytes);
    const uint32_t M = (uint32_t)M64, n = l.n;
    unsigned long long *cand = (unsigned long long *)(W + l.cand), *S = (unsigned long long *)(W + l.S);
    uint32_t *J = (uint32_t *)(W + l.J);
    if (M) {
        k_idx_scan<true><<<(unsigned)n_tiles, IDX_THREADS, 0, s>>>(buf, scan_len, marker_word, mb, nullptr, tile_base, cand);
        ambc_count_launch();
    }
    k_rng_link<<<(n + 255) / 256, 256, 0, s>>>(buf, rng_geo(r), cand, M, (IdxRec *)(W + l.rec), J, S);
    ambc_count_launch();
    for (int k = 1; k < l.K; k++) {
        k_rng_jump<<<(n + 255) / 256, 256, 0, s>>>(J + (uint64_t)(k - 1) * n, S + (uint64_t)(k - 1) * n, J + (uint64_t)k * n,
                                                    S + (uint64_t)k * n, n);
        ambc_count_launch();
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(s));
    return AMBC_OK;
}

// the fold step on the device; leaves the walk record in the info area
static int rng_fold(const ambc_range *r, const ambc_range_state *in, ambc_range_state *out, unsigned long long *walk,
                    cudaStream_t s)
{
    if (!r || !in || !r->work_dev) return ambc_fail(AMBC_E_ARG, "ambc_range: bad argument");
    const RngLayout l = rng_layout(r->hi - r->lo, r->n_cand);
    uint8_t *W = (uint8_t *)r->work_dev;
    ambc_range_state *d_in = (ambc_range_state *)(W + l.info + RNG_IN), *d_out = (ambc_range_state *)(W + l.info + RNG_OUT);
    unsigned long long *d_walk = (unsigned long long *)(W + l.info + RNG_WALK);
    CUDA_TRY(cudaMemcpyAsync(d_in, in, sizeof(ambc_range_state), cudaMemcpyHostToDevice, s));
    k_rng_fold<<<1, 1, 0, s>>>((const unsigned long long *)(W + l.cand), (const IdxRec *)(W + l.rec), (const uint32_t *)(W + l.J),
                               (const unsigned long long *)(W + l.S), l.n, l.K, (uint32_t)r->n_cand, rng_geo(r), d_in, d_out, d_walk);
    ambc_count_launch();
    CUDA_TRY(cudaGetLastError());
    if (out) CUDA_TRY(cudaMemcpyAsync(out, d_out, sizeof(ambc_range_state), cudaMemcpyDeviceToHost, s));
    if (walk) CUDA_TRY(cudaMemcpyAsync(walk, d_walk, 32, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return AMBC_OK;
}

extern "C" int ambc_range_fold(const ambc_range *r, const ambc_range_state *in, ambc_range_state *out, void *stream_)
{
    if (!out) return ambc_fail(AMBC_E_ARG, "ambc_range_fold: bad argument");
    return rng_fold(r, in, out, nullptr, (cudaStream_t)stream_);
}

extern "C" int ambc_range_table(const ambc_range *r, const ambc_range_state *entry, ambc_pkg *table_dev, uint64_t table_cap,
                                uint64_t *n_entries, uint64_t *out_lo, uint64_t *out_hi, uint64_t *need, void *stream_)
{
    cudaStream_t s = (cudaStream_t)stream_;
    if (n_entries) *n_entries = 0;
    if (need) *need = 0;
    ambc_range_state ex;
    unsigned long long walk[4] = {0, 0, 0, 0};
    int rc = rng_fold(r, entry, &ex, walk, s);
    if (rc) return rc;
    const RngGeo g = rng_geo(r);
    const uint64_t hdr = g.mb + 14, lo = g.lo;
    const uint64_t o_lo = rng_out_offset(*entry, lo, g.orig_size, g.mb, g.known_mask);
    if (out_lo) *out_lo = o_lo;
    if (out_hi) *out_hi = rng_out_offset(ex, g.hi, g.orig_size, g.mb, g.known_mask);
    // a copied-through package whose payload began in an earlier range
    uint64_t n_in = 0, in_pay = 0;
    RngShare in_sh = {0, 0};
    if (entry->pkg_pos != AMBC_RANGE_NO_PKG && rng_copied(entry->pkg_type, g.known_mask)) {
        in_pay = entry->pkg_pos + hdr;
        const uint64_t emit = rng_emit(rng_nominal(entry->pkg_type, g.known_mask, entry->pkg_comp, entry->pkg_orig), entry->pkg_out,
                                       g.orig_size);
        in_sh = rng_share(in_pay, entry->pkg_comp, emit, lo, g.hi, false);
        n_in = (in_sh.b - in_sh.a + IDX_RAW_PIECE - 1) / IDX_RAW_PIECE;
    }
    const uint64_t chain_len = walk[0];
    const RngLayout l = rng_layout(g.hi - lo, r->n_cand);
    uint8_t *W = (uint8_t *)r->work_dev;
    const IdxRec *rec = (const IdxRec *)(W + l.rec);
    const unsigned long long *cand = (const unsigned long long *)(W + l.cand);
    uint32_t *chain = (uint32_t *)(W + l.chain);
    unsigned long long *nominal = (unsigned long long *)(W + l.nom), *obefore = (unsigned long long *)(W + l.ob);
    unsigned long long *ecount = (unsigned long long *)(W + l.ec), *ebase = (unsigned long long *)(W + l.eb);
    unsigned long long *sct = (unsigned long long *)(W + l.sct), *tot = (unsigned long long *)(W + l.info + RNG_TOT);
    uint64_t n_chain = 0;
    const unsigned cgrid = (unsigned)((chain_len + 255) / 256);
    if (chain_len) {
        k_rng_chain<<<cgrid, 256, 0, s>>>((const uint32_t *)(W + l.J), l.n, l.K, (uint32_t)walk[1], chain_len, chain);
        k_idx_nominal<<<cgrid, 256, 0, s>>>(rec, chain, chain_len, g.known_mask, nominal);
        ambc_count_launch(); ambc_count_launch();
        if ((rc = dev_excl_scan(nominal, chain_len, obefore, sct, tot, s))) return rc;
        k_rng_entries<false><<<cgrid, 256, 0, s>>>(rec, chain, cand, nominal, obefore, chain_len, entry->out_before, g, ecount,
                                                    nullptr, 0, 0, nullptr);
        ambc_count_launch();
        if ((rc = dev_excl_scan(ecount, chain_len, ebase, sct, tot + 1, s))) return rc;
        unsigned long long h_tot = 0, h_last = 0;
        IdxRec last;
        CUDA_TRY(cudaMemcpyAsync(&h_tot, tot + 1, 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(&last, rec + walk[2], sizeof(IdxRec), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(&h_last, cand + walk[2], 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        n_chain = h_tot;
        // a decoded package needs its whole payload, also the part behind the halo
        if (need && last.kind == 0 && !rng_copied(last.type, g.known_mask) &&
            rng_emit(rng_nominal(last.type, g.known_mask, last.comp, last.orig), walk[3], g.orig_size)) {
            const uint64_t end = lo + h_last + hdr + last.comp, have = rng_min(g.hi + g.mb + 13, g.body_len);
            *need = end > have ? end - have : 0;
        }
    }
    const uint64_t ne = n_in + n_chain;
    if (n_entries) *n_entries = ne;
    if (table_dev && ne) {
        if (ne > table_cap) return ambc_fail(AMBC_E_CAPACITY, "ambc_range_table: table too small (%llu entries)", (unsigned long long)ne);
        if (n_in) {
            k_rng_inbound<<<(unsigned)((n_in + 255) / 256), 256, 0, s>>>(in_pay, entry->pkg_comp, in_sh, entry->pkg_out, lo, o_lo, table_dev);
            ambc_count_launch();
        }
        if (n_chain) {
            k_rng_entries<true><<<cgrid, 256, 0, s>>>(rec, chain, cand, nominal, obefore, chain_len, entry->out_before, g, nullptr,
                                                       ebase, n_in, o_lo, table_dev);
            ambc_count_launch();
        }
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaStreamSynchronize(s));
    }
    return AMBC_OK;
}
