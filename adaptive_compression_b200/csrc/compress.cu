// compress.cu -- chunk select / scan / pack kernels and the ambc_compress_* entry points.
//
// Replaces AdaptiveCompressor._adaptive_compress and its helpers
// (adaptive_compressor.py:363-394, 537-590, 595-700).
//
//   k_select_fast      one CTA per grid chunk (select_fast.cuh): gates, the exact size of every enabled
//                      candidate, the argmin in list order with the benefit test len+overhead < n, the
//                      winner's payload into its slot.
//   k_sizes / k_scan_tiles / k_offsets
//                      exclusive scan of package sizes with the "rest of file raw" rule: everything
//                      from the first chunk without a winner onward is ONE raw package.
//   k_pack             one CTA per chunk: 18-byte package header + payload to the final offset.
//   k_dynamic_walk     multi-candidate mode: the chain of chosen chunk sizes, walked segment by segment;
//                      k_select_span_fast / k_pack_span then encode and frame the chosen chunks.
#include "ambc_internal.h"
#include <vector>
#include "select_fast.cuh"


// select_fast.cuh: 128 threads and ~38 KB of shared memory per chunk, five CTAs per SM
template <int NMAX>
__global__ void __launch_bounds__(SF_T, NMAX <= 4096 ? 6 : 3)
k_select_fast(const uint8_t *__restrict__ in, uint64_t total, uint32_t N, uint32_t mask, uint32_t ovh,
              uint8_t *__restrict__ slots, uint64_t slot_stride, uint8_t *__restrict__ type,
              uint32_t *__restrict__ comp, unsigned long long *first_raw, uint64_t chunk_begin, uint64_t n_chunks,
              uint32_t strict)
{
    extern __shared__ uint4 smem4[];
    SfCtx<NMAX> c;
    sf_carve<NMAX>(c, (uint8_t *)smem4);
    for (uint64_t i = chunk_begin + blockIdx.x; i < n_chunks; i += gridDim.x) {
        const uint64_t off = i * (uint64_t)N;
        const int n = (int)min((uint64_t)N, total - off);
        // strict mode: a chunk behind a chunk without a winner lies inside the one raw package that ends the file
        // (adaptive_compressor.py:586-590), whatever its own trial would say.  first_raw only ever decreases, so a
        // value below i seen now is final enough: the scan and pack kernels ignore the map from first_raw on.
        // (one thread reads for the CTA: first_raw changes under the kernel's feet, and threads that read
        // different values would part ways in front of the barriers of the trial)
        if (strict) {
            if (threadIdx.x == 0) c.red[30] = *(volatile unsigned long long *)first_raw < i;
            __syncthreads();
        }
        if (strict && c.red[30]) {
            if (threadIdx.x == 0) { type[i] = 255; comp[i] = (uint32_t)n; }
            continue;
        }
        sf_load<NMAX>(c, in + off, n);
        const SfOut o = sf_select<NMAX>(c, mask, (int)ovh);
        __syncthreads();
        if (o.type != 255) {
            uint8_t *dst = slots + i * slot_stride; // 16-byte aligned
            const int nv = (o.len + 15) >> 4;
            for (int k = threadIdx.x; k < nv; k += SF_T) ((uint4 *)dst)[k] = ((const uint4 *)c.pay)[k];
        }
        if (threadIdx.x == 0) {
            type[i] = (uint8_t)o.type;
            comp[i] = (uint32_t)o.len;
            if (o.type == 255) atomicMin(first_raw, (unsigned long long)i);
        }
        __syncthreads();
    }
}

// span mode (multi-candidate path, see the span section below): chunks given by position and size
template <int NMAX>
__global__ void __launch_bounds__(SF_T, NMAX <= 4096 ? 6 : 3)
k_select_span_fast(const uint8_t *__restrict__ in, uint64_t total, uint32_t N, uint32_t mask, uint32_t ovh, uint32_t stride,
                   const unsigned long long *__restrict__ list, uint8_t *__restrict__ slots, uint8_t *__restrict__ type,
                   uint32_t *__restrict__ comp, uint64_t n_items)
{
    // list == nullptr: item i = [i * stride, i * stride + min(N, total - i * stride)), no payload kept;
    // else item i = (pos, size) = (list[2 i], low half of list[2 i + 1]) and its payload goes to slots + pos
    // (payloads are shorter than their chunks, so the chunk's own offset is a collision-free slot)
    extern __shared__ uint4 smem4[];
    SfCtx<NMAX> c;
    sf_carve<NMAX>(c, (uint8_t *)smem4);
    for (uint64_t i = blockIdx.x; i < n_items; i += gridDim.x) {
        uint64_t off;
        int n;
        if (list) { off = list[2 * i]; n = (int)(uint32_t)list[2 * i + 1]; }
        else { off = i * (uint64_t)stride; n = (int)min((uint64_t)N, total - off); }
        sf_load<NMAX>(c, in + off, n);
        const SfOut o = sf_select<NMAX>(c, mask, (int)ovh);
        __syncthreads();
        if (slots && o.type != 255) {
            uint8_t *dst = slots + off;
            if ((((uintptr_t)dst) & 15) == 0) {
                const int nv = (o.len + 15) >> 4;
                for (int k = threadIdx.x; k < nv; k += SF_T) ((uint4 *)dst)[k] = ((const uint4 *)c.pay)[k];
            } else {
                for (int k = threadIdx.x; k < o.len; k += SF_T) dst[k] = c.pay[k];
            }
        }
        if (threadIdx.x == 0) {
            type[i] = (uint8_t)o.type;
            comp[i] = (uint32_t)o.len;
        }
        __syncthreads();
    }
}

// ---- package-size scan ---------------------------------------------------------------------
// In strict mode chunks >= first_raw contribute nothing (they live inside the single raw
// package); in per-chunk-raw mode every chunk is its own package.
#define SCAN_TILE 2048
struct ScanState {
    unsigned long long first_raw;  // min chunk index without a winner, ~0 if none
    unsigned long long body_len;
    unsigned long long n_packages;
    unsigned long long payload_bytes;
    unsigned long long usage[5];
    unsigned long long carry;      // body bytes before the chunks not yet scanned (piece-wise runs)
};

__device__ __forceinline__ uint64_t pkg_size(uint64_t i, const uint8_t *type, const uint32_t *comp, uint32_t N,
                                             uint64_t total, uint32_t ovh, uint64_t first_raw, bool pcr)
{
    if (!pcr && i >= first_raw) return 0;
    uint64_t len = comp[i]; // raw chunks carry comp = n
    (void)N; (void)total; (void)type;
    return ovh + len;
}

__global__ void __launch_bounds__(256)
k_sizes(const uint8_t *__restrict__ type, const uint32_t *__restrict__ comp, uint64_t chunk_begin, uint64_t n_chunks,
        uint32_t N, uint64_t total, uint32_t ovh, uint32_t flags, const ScanState *st, unsigned long long *tile_sum)
{
    // chunks [chunk_begin, n_chunks); chunk_begin is a multiple of SCAN_TILE; tile_sum is indexed globally
    __shared__ unsigned long long red[8];
    const bool pcr = flags & 1u;
    const uint64_t fr = st->first_raw;
    uint64_t base = chunk_begin + (uint64_t)blockIdx.x * SCAN_TILE;
    unsigned long long s = 0;
    for (int k = threadIdx.x; k < SCAN_TILE; k += 256) {
        uint64_t i = base + k;
        if (i < n_chunks) s += pkg_size(i, type, comp, N, total, ovh, fr, pcr);
    }
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(FULL_MASK, s, d);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int i = 0; i < 8; i++) t += red[i];
        tile_sum[base / SCAN_TILE] = t;
    }
}

// single CTA: exclusive scan of the tile sums in place, body length, END package, stats
__global__ void __launch_bounds__(1024)
k_scan_tiles(unsigned long long *tile_sum, uint64_t tile_begin, uint64_t n_tiles, int is_last,
             const uint8_t *__restrict__ type, const uint32_t *__restrict__ comp, uint64_t n_chunks, uint32_t N,
             uint64_t total, uint32_t ovh, uint32_t flags, ScanState *st, uint8_t *out, uint64_t out_cap,
             uint32_t marker_word, uint32_t mb)
{
    // tiles [tile_begin, n_tiles), continuing from st->carry; the last call closes the body
    __shared__ unsigned long long wsum[32];
    __shared__ unsigned long long carry_s;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid == 0) carry_s = st->carry;
    __syncthreads();
    for (uint64_t base = tile_begin; base < n_tiles; base += 1024) {
        uint64_t i = base + tid;
        unsigned long long v = i < n_tiles ? tile_sum[i] : 0, inc = v;
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long t = __shfl_up_sync(FULL_MASK, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) wsum[w] = inc;
        __syncthreads();
        unsigned long long wbase = 0;
        for (int k = 0; k < w; k++) wbase += wsum[k];
        unsigned long long carry = carry_s;
        if (i < n_tiles) tile_sum[i] = carry + wbase + inc - v;
        __syncthreads();
        if (tid == 1023) carry_s = carry + wbase + inc;
        __syncthreads();
    }
    if (tid == 0) st->carry = carry_s;
    if (tid == 0 && is_last) {
        const bool pcr = flags & 1u;
        unsigned long long body = carry_s;
        unsigned long long fr = st->first_raw;
        unsigned long long npk = n_chunks;
        if (!pcr && fr != ~0ull) {
            // one raw package for the rest of the file (adaptive_compressor.py:586-590)
            body += ovh + (total - fr * (unsigned long long)N);
            npk = fr + 1;
        }
        st->n_packages = npk;
        if (!(flags & 2u)) { // (bit 1: the caller appends a raw tail package and END itself -- span mode)
            body += mb + 12; // END package (:595-607)
            if (body <= out_cap) {
                uint8_t *e = out + body - (mb + 12);
                for (uint32_t k = 0; k < mb; k++) e[k] = (uint8_t)(marker_word >> (8 * k));
                for (uint32_t k = 0; k < 12; k++) e[mb + k] = 0;
            }
        }
        st->body_len = body;
    }
}

__global__ void __launch_bounds__(256)
k_offsets(const uint8_t *__restrict__ type, const uint32_t *__restrict__ comp, uint64_t chunk_begin, uint64_t n_chunks,
          uint32_t N, uint64_t total, uint32_t ovh, uint32_t flags, ScanState *st,
          const unsigned long long *tile_base, unsigned long long *offs)
{
    // one tile per CTA, 8 chunks per thread
    __shared__ unsigned long long wsum[8];
    __shared__ unsigned long long ustat[6];
    const bool pcr = flags & 1u;
    const uint64_t fr = st->first_raw;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid < 6) ustat[tid] = 0;
    uint64_t base = chunk_begin + (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)tid * 8;
    unsigned long long v[8], s = 0;
    unsigned long long usage[5] = {0, 0, 0, 0, 0}, pbytes = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        uint64_t i = base + k;
        v[k] = i < n_chunks ? pkg_size(i, type, comp, N, total, ovh, fr, pcr) : 0;
        s += v[k];
        if (i < n_chunks && (pcr || i < fr)) {
            int t = type[i];
            if (t >= 1 && t <= 4) { usage[t]++; pbytes += comp[i]; }
            else usage[0]++;
        }
    }
    unsigned long long inc = s;
    for (int d = 1; d < 32; d <<= 1) {
        unsigned long long t = __shfl_up_sync(FULL_MASK, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    unsigned long long wbase = 0;
    for (int k = 0; k < w; k++) wbase += wsum[k];
    unsigned long long run = tile_base[chunk_begin / SCAN_TILE + blockIdx.x] + wbase + inc - s;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        uint64_t i = base + k;
        if (i < n_chunks) offs[i] = run;
        run += v[k];
    }
    // statistics (adaptive_compressor.py:471-480)
#pragma unroll
    for (int k = 0; k < 5; k++) {
        unsigned long long u = usage[k];
        for (int d = 16; d > 0; d >>= 1) u += __shfl_xor_sync(FULL_MASK, u, d);
        if (lane == 0 && u) atomicAdd(&ustat[k], u);
    }
    for (int d = 16; d > 0; d >>= 1) pbytes += __shfl_xor_sync(FULL_MASK, pbytes, d);
    if (lane == 0 && pbytes) atomicAdd(&ustat[5], pbytes);
    __syncthreads();
    if (tid < 5 && ustat[tid]) atomicAdd(&st->usage[tid], ustat[tid]);
    if (tid == 5 && ustat[5]) atomicAdd(&st->payload_bytes, ustat[5]);
}

// ---- pack ----------------------------------------------------------------------------------
// package header (adaptive_compressor.py:609-621): marker, type, k=0, used u32, orig u32, comp u32
__device__ __forceinline__ void write_pkg_header(uint8_t *h, uint32_t marker_word, uint32_t mb, int type,
                                                 uint32_t orig, uint32_t comp)
{
    for (uint32_t k = 0; k < mb; k++) h[k] = (uint8_t)(marker_word >> (8 * k));
    h[mb] = (uint8_t)type;
    h[mb + 1] = 0;
    store_u32le(h + mb + 2, orig);
    store_u32le(h + mb + 6, orig);
    store_u32le(h + mb + 10, comp);
}

#define PACK_BLOCK 128
__global__ void __launch_bounds__(PACK_BLOCK)
k_pack(const uint8_t *__restrict__ in, uint64_t total, uint32_t N, const uint8_t *__restrict__ slots,
       uint64_t slot_stride, const uint8_t *__restrict__ type, const uint32_t *__restrict__ comp,
       const unsigned long long *__restrict__ offs, const ScanState *st, uint32_t flags, uint32_t marker_word,
       uint32_t mb, uint8_t *__restrict__ out, uint64_t out_cap, uint64_t chunk_begin, uint64_t n_chunks, int check_cap)
{
    extern __shared__ uint4 smem4[];
    uint8_t *buf = (uint8_t *)smem4; // [32 header area][payload]
    const bool pcr = flags & 1u;
    const uint64_t fr = st->first_raw;
    const uint32_t ovh = mb + 14;
    if (check_cap && st->body_len > out_cap) return;
    for (uint64_t i = chunk_begin + blockIdx.x; i < n_chunks; i += gridDim.x) {
        uint64_t coff = i * (uint64_t)N;
        int n = (int)min((uint64_t)N, total - coff);
        if (!pcr && i >= fr) {
            // inside the single raw package: header once, then plain bytes
            uint64_t pbase = offs[fr]; // == offset of the raw package (sizes beyond fr are 0)
            uint64_t rawlen = total - fr * (uint64_t)N;
            copy_g2s<PACK_BLOCK>(buf + 32, in + coff, n);
            uint8_t *src = buf + 32;
            int len = n;
            if (i == fr) {
                if (threadIdx.x == 0) write_pkg_header(buf + 32 - ovh, marker_word, mb, 255, (uint32_t)rawlen, (uint32_t)rawlen);
                src = buf + 32 - ovh;
                len = n + ovh;
            }
            __syncthreads();
            uint64_t dst = (i == fr) ? pbase : pbase + ovh + (coff - fr * (uint64_t)N);
            copy_s2g<PACK_BLOCK>(out + dst, src, len);
        } else {
            int t = type[i];
            int len = (int)comp[i];
            if (t == 255) copy_g2s<PACK_BLOCK>(buf + 32, in + coff, n);
            else copy_g2s<PACK_BLOCK>(buf + 32, slots + i * slot_stride, len);
            if (threadIdx.x == 0) write_pkg_header(buf + 32 - ovh, marker_word, mb, t, (uint32_t)n, (uint32_t)len);
            __syncthreads();
            copy_s2g<PACK_BLOCK>(out + offs[i], buf + 32 - ovh, len + ovh);
        }
        __syncthreads();
    }
}

// ---- span mode: chunks given by (position, size) instead of the fixed grid ---------------------
// Used by the multi-candidate ("dynamic chunk size") path, adaptive_compressor.py:537-590, on the chosen
// chunk chain.  Separate kernels so that the fixed-grid hot path stays untouched.
struct ChunkSpan { unsigned long long pos; uint32_t size; uint32_t pad; };

static int launch_select_span(unsigned grid, cudaStream_t stream, const uint8_t *in, uint64_t total, uint32_t N,
                              uint32_t mask, uint32_t ovh, uint32_t stride, const ChunkSpan *list, uint8_t *slots,
                              uint8_t *type, uint32_t *comp, uint64_t n_items)
{
    static_assert(sizeof(ChunkSpan) == 16, "k_select_span_fast reads spans as two 64-bit words");
    if (N <= 4096) {
        CUDA_TRY(cudaFuncSetAttribute(k_select_span_fast<4096>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SfCfg<4096>::SMEM));
        k_select_span_fast<4096><<<grid, SF_T, SfCfg<4096>::SMEM, stream>>>(in, total, N, mask, ovh, stride, (const unsigned long long *)list,
                                                                            slots, type, comp, n_items);
    } else {
        CUDA_TRY(cudaFuncSetAttribute(k_select_span_fast<8192>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SfCfg<8192>::SMEM));
        k_select_span_fast<8192><<<grid, SF_T, SfCfg<8192>::SMEM, stream>>>(in, total, N, mask, ovh, stride, (const unsigned long long *)list,
                                                                            slots, type, comp, n_items);
    }
    ambc_count_launch();
    CUDA_TRY(cudaGetLastError());
    return AMBC_OK;
}

__global__ void __launch_bounds__(PACK_BLOCK)
k_pack_span(const uint8_t *__restrict__ in, const ChunkSpan *__restrict__ list, const uint8_t *__restrict__ slots,
            const uint8_t *__restrict__ type, const uint32_t *__restrict__ comp,
            const unsigned long long *__restrict__ offs, uint32_t marker_word, uint32_t mb,
            uint8_t *__restrict__ out, uint64_t n_items)
{
    extern __shared__ uint4 smem4[];
    uint8_t *buf = (uint8_t *)smem4; // [32 header area][payload]
    const uint32_t ovh = mb + 14;
    for (uint64_t i = blockIdx.x; i < n_items; i += gridDim.x) {
        const uint64_t coff = list[i].pos;
        const int n = (int)list[i].size;
        const int t = type[i];
        const int len = (int)comp[i];
        if (t == 255) {
            for (int k = threadIdx.x; k < n; k += PACK_BLOCK) buf[32 + k] = in[coff + k];
        } else {
            for (int k = threadIdx.x; k < len; k += PACK_BLOCK) buf[32 + k] = slots[coff + k];
        }
        if (threadIdx.x == 0) write_pkg_header(buf + 32 - ovh, marker_word, mb, t, (uint32_t)n, (uint32_t)len);
        __syncthreads();
        copy_s2g<PACK_BLOCK>(out + offs[i], buf + 32 - ovh, len + ovh);
        __syncthreads();
    }
}

// ---- host side -----------------------------------------------------------------------------
struct WorkLayout {
    uint64_t slots, type, comp, offs, tiles, state, total;
    uint64_t slot_stride, n_chunks, n_tiles;
};
static WorkLayout work_layout(uint64_t n, uint32_t chunk)
{
    WorkLayout L;
    L.n_chunks = chunk ? (n + chunk - 1) / chunk : 0;
    L.n_tiles = (L.n_chunks + SCAN_TILE - 1) / SCAN_TILE;
    L.slot_stride = chunk <= AMBC_NMAX ? ((uint64_t)chunk + 15) & ~15ull : 0;
    uint64_t o = 0;
    auto take = [&](uint64_t bytes) { uint64_t r = o; o += (bytes + 255) & ~255ull; return r; };
    L.slots = take(L.n_chunks * L.slot_stride + 16);
    L.type = take(L.n_chunks + 16);
    L.comp = take(L.n_chunks * 4 + 16);
    L.offs = take(L.n_chunks * 8 + 16);
    L.tiles = take(L.n_tiles * 8 + 16);
    L.state = take(sizeof(ScanState));
    L.total = o;
    return L;
}

extern "C" uint64_t ambc_compress_workspace_bytes(uint64_t n, uint32_t chunk)
{
    return work_layout(n, chunk).total;
}

extern "C" uint64_t ambc_compress_bound(uint64_t n, uint32_t chunk, uint32_t marker_bytes)
{
    uint64_t chunks = chunk ? (n + chunk - 1) / chunk : 0;
    return n + (chunks + 1) * (marker_bytes + 14) + marker_bytes + 12 + 64;
}

// piece_ready[k] (optional): event after which chunks [piece_start[k], piece_start[k + 1]) of the input
// are resident (ambc_compress_host uploads piece-wise so that H2D overlaps k_select); piece_start has
// n_pieces + 1 ascending entries, multiples of SCAN_TILE, the last one >= the chunk count
int ambc_compress_dev_impl(const void *in_dev, uint64_t n, uint32_t chunk, uint32_t method_mask, uint32_t flags,
                           const uint8_t *marker, uint32_t marker_bytes, void *out_dev, uint64_t out_cap,
                           void *work_dev, uint64_t work_bytes, ambc_compress_result *res, cudaStream_t stream,
                           const cudaEvent_t *piece_ready, const uint64_t *piece_start, uint32_t n_pieces,
                           const AmbcPieceOut *po);
extern "C" uint64_t ambc_scan_state_bytes(void) { return sizeof(ScanState); }

extern "C" int ambc_compress_dev(const void *in_dev, uint64_t n, uint32_t chunk, uint32_t method_mask,
                                 uint32_t flags, const uint8_t *marker, uint32_t marker_bytes, void *out_dev,
                                 uint64_t out_cap, void *work_dev, uint64_t work_bytes, ambc_compress_result *res,
                                 void *stream_)
{
    return ambc_compress_dev_impl(in_dev, n, chunk, method_mask, flags, marker, marker_bytes, out_dev, out_cap, work_dev,
                                  work_bytes, res, (cudaStream_t)stream_, nullptr, nullptr, 0, nullptr);
}

int ambc_compress_dev_impl(const void *in_dev, uint64_t n, uint32_t chunk, uint32_t method_mask, uint32_t flags,
                           const uint8_t *marker, uint32_t marker_bytes, void *out_dev, uint64_t out_cap,
                           void *work_dev, uint64_t work_bytes, ambc_compress_result *res, cudaStream_t stream,
                           const cudaEvent_t *piece_ready, const uint64_t *piece_start, uint32_t n_pieces,
                           const AmbcPieceOut *po)
{
    if (!res || !marker || marker_bytes < 1 || marker_bytes > 4 || chunk == 0)
        return ambc_fail(AMBC_E_ARG, "ambc_compress_dev: bad argument");
    if ((n && (!in_dev || !work_dev)) || !out_dev) return ambc_fail(AMBC_E_ARG, "ambc_compress_dev: null buffer");
    WorkLayout L = work_layout(n, chunk);
    if (work_bytes < L.total) return ambc_fail(AMBC_E_CAPACITY, "ambc_compress_dev: workspace too small");
    if ((uint64_t)chunk > 0xFFFFFFFFull - 32) return ambc_fail(AMBC_E_ARG, "chunk too large");
    uint32_t ovh = marker_bytes + 14;
    uint32_t marker_word = 0;
    for (uint32_t k = 0; k < marker_bytes; k++) marker_word |= (uint32_t)marker[k] << (8 * k);
    memset(res, 0, sizeof(*res));
    res->n_chunks = L.n_chunks;
    res->map_type_off = L.type;
    res->map_comp_off = L.comp;

    uint8_t *W = (uint8_t *)work_dev;
    ScanState *st = (ScanState *)(W + L.state);
    ScanState h_st;
    memset(&h_st, 0, sizeof h_st);
    h_st.first_raw = ~0ull;

    if (n == 0) { // only the END package
        uint8_t endp[16];
        memcpy(endp, marker, marker_bytes);
        memset(endp + marker_bytes, 0, 12);
        if (out_cap < marker_bytes + 12) return ambc_fail(AMBC_E_CAPACITY, "out too small");
        CUDA_TRY(cudaMemcpyAsync(out_dev, endp, marker_bytes + 12, cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        if (po && po->out_host) {
            if (po->out_cap < marker_bytes + 12) return ambc_fail(AMBC_E_CAPACITY, "ambc_compress_host: out_cap too small");
            memcpy(po->out_host, endp, marker_bytes + 12);
        }
        res->body_len = marker_bytes + 12;
        res->first_raw = -1;
        return AMBC_OK;
    }
    // chunks of more than 4 GiB cannot be framed (u32 length fields, :617-619)
    bool native = chunk <= AMBC_NMAX && (method_mask & AMBC_NATIVE_MASK);
    if (!native) h_st.first_raw = 0; // no native method is eligible: everything is raw
    CUDA_TRY(cudaMemcpyAsync(st, &h_st, sizeof h_st, cudaMemcpyHostToDevice, stream));

    uint8_t *type = W + L.type;
    uint32_t *comp = (uint32_t *)(W + L.comp);
    unsigned long long *offs = (unsigned long long *)(W + L.offs);
    unsigned long long *tiles = (unsigned long long *)(W + L.tiles);
    unsigned grid_chunks = (unsigned)min<uint64_t>(L.n_chunks, 0x7fffffffull);

    if (native) {
        size_t psmem = 32 + (((size_t)chunk + 15) & ~(size_t)15) + 32;
        CUDA_TRY(cudaFuncSetAttribute(k_pack, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem));
        CUDA_TRY(cudaFuncSetAttribute(k_select_fast<4096>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SfCfg<4096>::SMEM));
        CUDA_TRY(cudaFuncSetAttribute(k_select_fast<8192>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SfCfg<8192>::SMEM));
        // piece-wise run (host-buffer path): select / scan / pack of piece k are queued behind the
        // upload of piece k; the finished body bytes of a piece go home while later pieces compute
        bool pieces = piece_ready && n_pieces > 1 && piece_start && piece_start[0] == 0 && piece_start[n_pieces] >= L.n_chunks;
        for (uint32_t k = 0; pieces && k < n_pieces; k++)
            pieces = piece_start[k] % SCAN_TILE == 0 && piece_start[k] < piece_start[k + 1];
        if (!pieces && piece_ready)
            for (uint32_t k = 0; k < n_pieces; k++) CUDA_TRY(cudaStreamWaitEvent(stream, piece_ready[k], 0));
        const uint32_t np = pieces ? n_pieces : 1;
        const bool stream_out = pieces && po && po->out_host && po->states && po->done;
        cudaStream_t s2 = (stream_out && po->aux && po->sel) ? po->aux : stream;
        for (uint32_t k = 0; k < np; k++) {
            const uint64_t c0 = pieces ? piece_start[k] : 0;
            const uint64_t c1 = pieces ? min<uint64_t>(L.n_chunks, piece_start[k + 1]) : L.n_chunks;
            if (c0 >= c1) break;
            const bool last = c1 == L.n_chunks;
            const unsigned gch = (unsigned)min<uint64_t>(c1 - c0, 0x7fffffffull);
            const unsigned gt = (unsigned)((c1 - c0 + SCAN_TILE - 1) / SCAN_TILE);
            if (pieces) CUDA_TRY(cudaStreamWaitEvent(stream, piece_ready[k], 0));
            if (k == 0) ambc_timing_mark(0, stream);
            if (chunk <= 4096)
                k_select_fast<4096><<<gch, SF_T, SfCfg<4096>::SMEM, stream>>>((const uint8_t *)in_dev, n, chunk, method_mask, ovh,
                                                                             W + L.slots, L.slot_stride, type, comp,
                                                                             &st->first_raw, c0, c1, (flags & AMBC_F_PER_CHUNK_RAW) ? 0u : 1u);
            else
                k_select_fast<8192><<<gch, SF_T, SfCfg<8192>::SMEM, stream>>>((const uint8_t *)in_dev, n, chunk, method_mask, ovh,
                                                                             W + L.slots, L.slot_stride, type, comp,
                                                                             &st->first_raw, c0, c1, (flags & AMBC_F_PER_CHUNK_RAW) ? 0u : 1u);
            ambc_count_launch();
            if (last) ambc_timing_mark(1, stream);
            // scan + pack of piece k run on their own stream so that k_select of piece k + 1 follows at once
            // (k_select only lowers st->first_raw to chunks of its own piece, which the scans of earlier
            // pieces never look at)
            if (s2 != stream) {
                CUDA_TRY(cudaEventRecord(po->sel[k], stream));
                CUDA_TRY(cudaStreamWaitEvent(s2, po->sel[k], 0));
            }
            k_sizes<<<gt, 256, 0, s2>>>(type, comp, c0, c1, chunk, n, ovh, flags, st, tiles);
            ambc_count_launch();
            k_scan_tiles<<<1, 1024, 0, s2>>>(tiles, c0 / SCAN_TILE, (c1 + SCAN_TILE - 1) / SCAN_TILE, last ? 1 : 0, type,
                                             comp, L.n_chunks, chunk, n, ovh, flags, st, (uint8_t *)out_dev, out_cap,
                                             marker_word, marker_bytes);
            ambc_count_launch();
            k_offsets<<<gt, 256, 0, s2>>>(type, comp, c0, c1, chunk, n, ovh, flags, st, tiles, offs);
            ambc_count_launch();
            if (last) ambc_timing_mark(2, s2);
            k_pack<<<gch, PACK_BLOCK, psmem, s2>>>((const uint8_t *)in_dev, n, chunk, W + L.slots, L.slot_stride, type,
                                                   comp, offs, st, flags, marker_word, marker_bytes, (uint8_t *)out_dev,
                                                   out_cap, c0, c1, pieces ? 0 : 1);
            ambc_count_launch();
            CUDA_TRY(cudaGetLastError());
            if (stream_out) {
                CUDA_TRY(cudaMemcpyAsync((uint8_t *)po->states + (size_t)k * sizeof(ScanState), st, sizeof(ScanState),
                                         cudaMemcpyDeviceToHost, s2));
                CUDA_TRY(cudaEventRecord(po->done[k], s2));
                if (last && s2 != stream) CUDA_TRY(cudaStreamWaitEvent(stream, po->done[k], 0));
            }
        }
        ambc_timing_mark(3, stream);
        ambc_timing().pending_c = ambc_timing().on;
        uint64_t sent = 0;
        if (stream_out) {
            // bytes [sent, carry_k) are final after piece k as long as no chunk lacked a winner
            for (uint32_t k = 0; k + 1 < np; k++) {
                CUDA_TRY(cudaEventSynchronize(po->done[k]));
                const ScanState *hs = (const ScanState *)((const uint8_t *)po->states + (size_t)k * sizeof(ScanState));
                if (hs->first_raw != ~0ull || hs->carry > po->out_cap) break;
                if (hs->carry > sent) {
                    CUDA_TRY(cudaMemcpyAsync((uint8_t *)po->out_host + sent, (const uint8_t *)out_dev + sent, hs->carry - sent,
                                             cudaMemcpyDeviceToHost, po->d2h));
                    sent = hs->carry;
                }
            }
        }
        CUDA_TRY(cudaMemcpyAsync(&h_st, st, sizeof h_st, cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        if (po && po->out_host) {
            if (h_st.body_len > po->out_cap || h_st.body_len > out_cap) {
                cudaStreamSynchronize(po->d2h);
                return ambc_fail(AMBC_E_CAPACITY, "ambc_compress_host: out_cap %llu < body %llu",
                                 (unsigned long long)po->out_cap, (unsigned long long)h_st.body_len);
            }
            CUDA_TRY(cudaMemcpyAsync((uint8_t *)po->out_host + sent, (const uint8_t *)out_dev + sent, h_st.body_len - sent,
                                     cudaMemcpyDeviceToHost, stream));
            CUDA_TRY(cudaStreamSynchronize(stream));
            CUDA_TRY(cudaStreamSynchronize(po->d2h));
        }
    } else {
        // one raw package: header + memcpy + END, no kernel needed beyond the copy engine
        if (piece_ready)
            for (uint32_t k = 0; k < n_pieces; k++) CUDA_TRY(cudaStreamWaitEvent(stream, piece_ready[k], 0));
        uint64_t body = (uint64_t)ovh + n + marker_bytes + 12;
        if (n > 0xFFFFFFFFull) return ambc_fail(AMBC_E_ARG, "raw package over 4 GiB cannot be framed (u32 fields)");
        if (body > out_cap) return ambc_fail(AMBC_E_CAPACITY, "out too small");
        uint8_t hdr[18], endp[16];
        memcpy(hdr, marker, marker_bytes);
        hdr[marker_bytes] = 255; hdr[marker_bytes + 1] = 0;
        uint32_t n32 = (uint32_t)n;
        for (int r = 0; r < 3; r++) memcpy(hdr + marker_bytes + 2 + 4 * r, &n32, 4);
        memcpy(endp, marker, marker_bytes);
        memset(endp + marker_bytes, 0, 12);
        uint8_t *o = (uint8_t *)out_dev;
        CUDA_TRY(cudaMemcpyAsync(o, hdr, ovh, cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(o + ovh, in_dev, n, cudaMemcpyDeviceToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(o + ovh + n, endp, marker_bytes + 12, cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemsetAsync(type, 255, L.n_chunks, stream));
        if (po && po->out_host) {
            if (body > po->out_cap) return ambc_fail(AMBC_E_CAPACITY, "ambc_compress_host: out_cap too small");
            CUDA_TRY(cudaMemcpyAsync(po->out_host, out_dev, body, cudaMemcpyDeviceToHost, stream));
        }
        CUDA_TRY(cudaStreamSynchronize(stream));
        h_st.body_len = body;
        h_st.n_packages = 1;
        h_st.usage[0] = 1;
    }
    if (h_st.body_len > out_cap) return ambc_fail(AMBC_E_CAPACITY, "ambc_compress_dev: out_cap too small");
    // the rest-of-file raw package carries its length in u32 fields (adaptive_compressor.py:617-619)
    if (native && !(flags & AMBC_F_PER_CHUNK_RAW) && h_st.first_raw != ~0ull &&
        n - h_st.first_raw * (uint64_t)chunk > 0xFFFFFFFFull)
        return ambc_fail(AMBC_E_ARG, "raw package over 4 GiB cannot be framed (u32 fields)");
    res->body_len = h_st.body_len;
    res->first_raw = h_st.first_raw == ~0ull ? -1 : (int64_t)h_st.first_raw;
    res->n_packages = h_st.n_packages;
    res->payload_bytes = h_st.payload_bytes;
    for (int k = 0; k < 5; k++) res->usage[k] = h_st.usage[k];
    if (native && !(flags & AMBC_F_PER_CHUNK_RAW) && res->first_raw >= 0) res->usage[0] = 1;
    return AMBC_OK;
}

#ifdef AMBC_PHASE_TIMING
extern "C" int ambc_sf_phase_read(unsigned long long *out48, int reset)
{
    cudaMemcpyFromSymbol(out48, g_sf, sizeof(unsigned long long) * 48);
    if (reset) { unsigned long long z[48] = {0}; cudaMemcpyToSymbol(g_sf, z, sizeof z); }
    return 0;
}
#endif
// ---- multi-candidate ("dynamic chunk size") mode ------------------------------------------------
// adaptive_compressor.py:537-590 with several CHUNK_SIZE_CANDIDATES: at every position each candidate
// size (clamped to the remaining bytes) is tried, the smallest ratio (len + overhead) / size wins,
// larger candidates win ties; no winner -> the rest of the file is one raw package.
// Every reachable position is a multiple of g = gcd(candidates).  The chain is walked on the GPU
// (k_dynamic_walk, below), and the chosen chunks are encoded and framed in span mode.
static uint64_t gcd64(uint64_t a, uint64_t b) { while (b) { uint64_t t = a % b; a = b; b = t; } return a; }

// ---- the chain of the multi-candidate mode on the GPU ---------------------------------------------------------
// The reference walks the file once: at every position it tries every candidate size and moves on by the winner's
// size (adaptive_compressor.py:363-394, 537-590).  Only the positions on that chain matter, about one in six of
// the multiples of g.  The file is cut into segments of DYN_SEGU * g bytes; one CTA walks the chain of a segment
// from its first byte, evaluating the candidates at the positions it actually visits (speculative: the true chain
// may enter the segment elsewhere).  Chains that enter a segment at different positions meet after a few packages
// (the winner at a position is a function of the position), so the host stitches the true chain from the
// speculative ones and re-enters (a second launch, same kernel) only the segments whose true entry differs, each
// until it meets the segment's speculative chain.
#define DYN_SEGU 64
struct WalkRec { unsigned long long pos; uint32_t size; uint32_t type_len; };   // type << 24 | payload length
struct WalkSeg { unsigned long long exit; unsigned long long stop; uint32_t count; uint32_t merged; uint32_t pad[2]; };
struct WalkCands { uint32_t n; uint32_t c[32]; };
// PER_ITEM = false: ambc_compress_dynamic_dev; true: the list-mode walks of ambc_dyn_range_* (a range's candidate
// entries all lie in its segment 0, so their records are stored per item)
template <bool PER_ITEM>
__global__ void __launch_bounds__(SF_T, 3)
k_dynamic_walk(const uint8_t *__restrict__ in, uint64_t total, WalkCands cands, uint32_t mask, uint32_t ovh, uint32_t pcr,
               uint32_t g, const unsigned long long *__restrict__ list, uint64_t n_items,
               const WalkRec *__restrict__ spec_recs, const WalkSeg *__restrict__ spec_segs,
               WalkRec *__restrict__ recs, WalkSeg *__restrict__ segs)
{
    // list == nullptr: item i = segment i entered at its first byte; else item i = (segment, entry position) and the
    // walk stops where it meets the segment's speculative chain (spec_recs / spec_segs).  Records go to
    // recs[segment * DYN_SEGU], or with PER_ITEM to recs[item * DYN_SEGU] (several items may share a segment)
    extern __shared__ uint4 smem4[];
    SfCtx<8192> c;
    sf_carve<8192>(c, (uint8_t *)smem4);
    __shared__ uint32_t visited[DYN_SEGU / 32];
    const uint64_t seglen = (uint64_t)DYN_SEGU * g;
    for (uint64_t it = blockIdx.x; it < n_items; it += gridDim.x) {
        const uint64_t sg = list ? list[2 * it] : it;
        const uint64_t s0 = sg * seglen, s1 = min(total, s0 + seglen);
        uint64_t pos = list ? list[2 * it + 1] : s0;
        if (list) { // positions the speculative chain of this segment visits
            if (threadIdx.x < DYN_SEGU / 32) visited[threadIdx.x] = 0;
            __syncthreads();
            const uint32_t cnt = spec_segs[sg].count;
            for (uint32_t k = threadIdx.x; k < cnt; k += SF_T) {
                const uint32_t u = (uint32_t)((spec_recs[sg * DYN_SEGU + k].pos - s0) / g);
                atomicOr(&visited[u >> 5], 1u << (u & 31));
            }
            __syncthreads();
        }
        uint32_t count = 0, merged = 0;
        unsigned long long stop = ~0ull;
        while (pos < s1) {
            if (list) {
                const uint32_t u = (uint32_t)((pos - s0) / g);
                if ((visited[u >> 5] >> (u & 31)) & 1u) { merged = 1; break; }
            }
            const uint64_t remain = total - pos;
            // (adaptive_compressor.py:548-584) every candidate, clamped to the rest of the file, in list order; the
            // smallest (len + overhead) / size wins as a double, the first of equals stays
            double best_ratio = 1.0;
            uint32_t best_c = 0, best_t = 255, best_len = 0, last_c = 0, last_t = 255, last_len = 0;
            for (uint32_t ci = 0; ci < cands.n; ci++) {
                const uint32_t cs = (uint64_t)cands.c[ci] < remain ? cands.c[ci] : (uint32_t)remain;
                if (cs > AMBC_NMAX) continue; // no native method is eligible (:114-127)
                uint32_t t, len;
                if (cs == last_c) { t = last_t; len = last_len; } // (clamped candidates repeat near the end of the file)
                else {
                    sf_load<8192>(c, in + pos, (int)cs);
                    const SfOut o = sf_select<8192>(c, mask, (int)ovh);
                    __syncthreads();
                    t = (uint32_t)o.type; len = (uint32_t)o.len;
                    last_c = cs; last_t = t; last_len = len;
                }
                if (t == 255) continue;
                const double ratio = (double)((uint64_t)len + ovh) / (double)cs;
                if (ratio < best_ratio) { best_ratio = ratio; best_c = cs; best_t = t; best_len = len; }
            }
            if (best_t == 255) {
                if (!pcr) { stop = pos; break; } // rest of the file raw (:586-590)
                best_c = (uint64_t)cands.c[cands.n - 1] < remain ? cands.c[cands.n - 1] : (uint32_t)remain; // labelled extension
                best_len = best_c;
            }
            if (threadIdx.x == 0) {
                WalkRec r;
                r.pos = pos; r.size = best_c; r.type_len = (best_t << 24) | best_len;
                recs[(PER_ITEM ? it : sg) * DYN_SEGU + count] = r;
            }
            count++;
            pos += best_c;
        }
        if (threadIdx.x == 0) {
            WalkSeg w;
            w.exit = pos; w.stop = stop; w.count = count; w.merged = merged; w.pad[0] = w.pad[1] = 0;
            segs[list ? it : sg] = w;
        }
        __syncthreads();
    }
}

struct DynLayout {
    uint64_t slots, spans, type, comp, offs, tiles, state, walk_recs, walk_segs, walk_list, total;
    uint64_t n_pos, n_tiles, g, n_seg;
};
// n: the bytes whose chain is walked (the file, or a range [lo, hi)); items > 0: a range, whose list-mode walks store
// their records per item (up to `items` of them) and whose last packages may run up to 8192 bytes past its end
static int dyn_layout(uint64_t n, const uint32_t *cands, uint32_t n_cands, DynLayout &L, uint64_t items = 0)
{
    if (!cands || n_cands < 1 || n_cands > 32) return ambc_fail(AMBC_E_ARG, "need 1..32 candidate sizes");
    uint64_t g = 0;
    for (uint32_t i = 0; i < n_cands; i++) {
        if (cands[i] == 0) return ambc_fail(AMBC_E_ARG, "candidate size 0");
        if (i && cands[i] >= cands[i - 1]) return ambc_fail(AMBC_E_ARG, "candidate sizes must be strictly descending");
        g = gcd64(g, cands[i]);
    }
    if (g < 256 || g % 16) return ambc_fail(AMBC_E_ARG, "candidate sizes need a common divisor that is a multiple of 16 and >= 256");
    L.g = g;
    L.n_pos = (n + g - 1) / g;
    // sizes clamped to 8192 (candidates are strictly descending, so equal clamped sizes are adjacent)
    uint32_t n_sizes = 0;
    for (uint32_t i = 0; i < n_cands; i++)
        if (!i || min(cands[i], (uint32_t)AMBC_NMAX) != min(cands[i - 1], (uint32_t)AMBC_NMAX)) n_sizes++;
    if (n_sizes > 16) return ambc_fail(AMBC_E_ARG, "too many distinct candidate sizes");
    L.n_tiles = (L.n_pos + SCAN_TILE - 1) / SCAN_TILE;
    uint64_t o = 0;
    auto take = [&](uint64_t bytes) { uint64_t r = o; o += (bytes + 255) & ~255ull; return r; };
    L.slots = take(n + (items ? AMBC_NMAX : 0) + 64);
    L.spans = take(L.n_pos * sizeof(ChunkSpan) + 16);
    L.type = take(L.n_pos + 16);
    L.comp = take(L.n_pos * 4 + 16);
    L.offs = take(L.n_pos * 8 + 16);
    L.tiles = take(L.n_tiles * 8 + 16);
    L.state = take(sizeof(ScanState));
    L.n_seg = (L.n_pos + DYN_SEGU - 1) / DYN_SEGU;
    L.walk_recs = take((L.n_pos + (items ? items * DYN_SEGU : L.n_pos)) * sizeof(WalkRec) + 64); // speculative | re-entered
    L.walk_segs = take((L.n_seg + (items ? items : L.n_seg)) * sizeof(WalkSeg) + 64);
    L.walk_list = take((items ? items : L.n_seg) * 16 + 64);
    L.total = o;
    return AMBC_OK;
}

extern "C" uint64_t ambc_compress_dynamic_workspace_bytes(uint64_t n, const uint32_t *cands, uint32_t n_cands)
{
    DynLayout L;
    if (dyn_layout(n, cands, n_cands, L)) return 0;
    return L.total;
}

// ---- the chain stitch of one walked span: the whole file, or a range [lo, hi) with positions relative to lo --------
struct DynStitch {
    const uint8_t *in;
    uint64_t total, len;  // bytes from position 0 to the end of the file; bytes whose chain is walked
    WalkCands wc;
    uint32_t mask, ovh, pcr;
    bool per_item;        // list-mode walks store their records per item (k_dynamic_walk<true>)
    uint64_t g, seglen, n_seg, n_pos;
    WalkRec *d_spec, *d_fix;
    WalkSeg *d_sseg, *d_fseg;
    unsigned long long *d_list;
    std::vector<WalkRec> h_spec, h_fix;
    std::vector<WalkSeg> h_sseg, fixseg;
    std::vector<uint64_t> fix_entry; // entry position the stored re-entered chain of a segment belongs to
    std::vector<WalkRec> extra_recs; // the walks of the extra items of the first round (a range's candidate entries)
    std::vector<WalkSeg> extra_segs;
};

static void dyn_stitch_init(DynStitch &S, const void *in, uint64_t total, uint64_t len, const uint32_t *cands,
                            uint32_t n_cands, uint32_t mask, uint32_t ovh, bool pcr, bool per_item, const DynLayout &L,
                            uint8_t *W)
{
    S.in = (const uint8_t *)in;
    S.total = total; S.len = len;
    S.wc.n = n_cands;
    for (uint32_t i = 0; i < n_cands; i++) S.wc.c[i] = cands[i];
    S.mask = mask; S.ovh = ovh; S.pcr = pcr ? 1u : 0u; S.per_item = per_item;
    S.g = L.g; S.seglen = (uint64_t)DYN_SEGU * L.g; S.n_seg = L.n_seg; S.n_pos = L.n_pos;
    S.d_spec = (WalkRec *)(W + L.walk_recs); S.d_fix = S.d_spec + L.n_pos;
    S.d_sseg = (WalkSeg *)(W + L.walk_segs); S.d_fseg = S.d_sseg + L.n_seg;
    S.d_list = (unsigned long long *)(W + L.walk_list);
    S.h_spec.assign(L.n_pos, WalkRec());
    S.h_fix.assign(L.n_pos, WalkRec());
    S.h_sseg.assign(L.n_seg, WalkSeg());
    S.fixseg.assign(L.n_seg, WalkSeg());
    S.fix_entry.assign(L.n_seg, ~0ull);
}

static int dyn_launch(const DynStitch &S, const unsigned long long *list, uint64_t n_items, WalkRec *recs, WalkSeg *segs,
                      cudaStream_t stream)
{
    const size_t wsmem = SfCfg<8192>::SMEM;
    const unsigned grid = (unsigned)min<uint64_t>(n_items, 0x7fffffffull);
    const WalkRec *sr = list ? S.d_spec : nullptr;
    const WalkSeg *ss = list ? S.d_sseg : nullptr;
    if (list && S.per_item) {
        CUDA_TRY(cudaFuncSetAttribute(k_dynamic_walk<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
        k_dynamic_walk<true><<<grid, SF_T, wsmem, stream>>>(S.in, S.total, S.wc, S.mask, S.ovh, S.pcr, (uint32_t)S.g, list,
                                                            n_items, sr, ss, recs, segs);
    } else {
        CUDA_TRY(cudaFuncSetAttribute(k_dynamic_walk<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
        k_dynamic_walk<false><<<grid, SF_T, wsmem, stream>>>(S.in, S.total, S.wc, S.mask, S.ovh, S.pcr, (uint32_t)S.g, list,
                                                             n_items, sr, ss, recs, segs);
    }
    ambc_count_launch();
    CUDA_TRY(cudaGetLastError());
    return AMBC_OK;
}

// the speculative chain of every segment, entered at its first byte
static int dyn_spec_walk(DynStitch &S, cudaStream_t stream)
{
    int rc = dyn_launch(S, nullptr, S.n_seg, S.d_spec, S.d_sseg, stream);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(S.h_spec.data(), S.d_spec, S.n_pos * sizeof(WalkRec), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaMemcpyAsync(S.h_sseg.data(), S.d_sseg, S.n_seg * sizeof(WalkSeg), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    return AMBC_OK;
}

// follows the chain from e through the segments with what is known and appends the (segment, entry) pairs that still
// have to be walked (unknown ones are assumed to meet their speculative chain).  With none appended, *exit (the first
// position at or past len) or *stop (no winner there, strict mode) is where the chain leaves the span.
static void dyn_follow(const DynStitch &S, uint64_t e, std::vector<unsigned long long> &list, uint64_t *exit, uint64_t *stop)
{
    *stop = ~0ull;
    for (uint64_t sg = e / S.seglen; sg < S.n_seg && e < S.len; sg++) {
        const uint64_t s0 = sg * S.seglen, s1 = min<uint64_t>(S.len, s0 + S.seglen);
        if (e >= s1) continue;
        const WalkSeg &sp = S.h_sseg[sg];
        if (e == s0) { if (sp.stop != ~0ull) { *stop = sp.stop; break; } e = sp.exit; continue; }
        if (S.fix_entry[sg] == e) {
            const WalkSeg &last = S.fixseg[sg].merged ? sp : S.fixseg[sg];
            if (last.stop != ~0ull) { *stop = last.stop; break; }
            e = last.exit;
            continue;
        }
        list.push_back(sg); list.push_back(e);
        if (sp.stop != ~0ull) { *stop = sp.stop; break; }
        e = sp.exit;
    }
    *exit = e;
}

// re-enters segments (one launch per round) until the chain from e0 is known to where it leaves the span; the first
// round also walks `extra` (segment, entry) items, whose records land in S.extra_recs / S.extra_segs
static int dyn_stitch(DynStitch &S, uint64_t e0, const std::vector<unsigned long long> &extra, uint64_t *exit,
                      uint64_t *stop, cudaStream_t stream)
{
    std::vector<unsigned long long> list;
    std::vector<WalkSeg> h_fseg;
    std::vector<WalkRec> h_items;
    for (int round = 0;; round++) {
        list.clear();
        dyn_follow(S, e0, list, exit, stop);
        const uint64_t n_local = list.size() / 2;
        if (round == 0) list.insert(list.end(), extra.begin(), extra.end());
        if (list.empty()) break;
        if (round > (int)S.n_seg + 2) return ambc_fail(AMBC_E_CUDA, "internal: the chain stitch does not settle");
        const uint64_t ni = list.size() / 2;
        CUDA_TRY(cudaMemcpyAsync(S.d_list, list.data(), list.size() * 8, cudaMemcpyHostToDevice, stream));
        int rc = dyn_launch(S, S.d_list, ni, S.d_fix, S.d_fseg, stream);
        if (rc) return rc;
        h_fseg.resize(ni);
        CUDA_TRY(cudaMemcpyAsync(h_fseg.data(), S.d_fseg, ni * sizeof(WalkSeg), cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        if (S.per_item) {
            h_items.resize(ni * DYN_SEGU);
            CUDA_TRY(cudaMemcpyAsync(h_items.data(), S.d_fix, ni * DYN_SEGU * sizeof(WalkRec), cudaMemcpyDeviceToHost, stream));
            CUDA_TRY(cudaStreamSynchronize(stream));
            for (uint64_t k = 0; k < n_local; k++)
                std::copy(h_items.begin() + k * DYN_SEGU, h_items.begin() + k * DYN_SEGU + h_fseg[k].count,
                          S.h_fix.begin() + list[2 * k] * DYN_SEGU);
            if (round == 0 && ni > n_local) {
                S.extra_recs.assign(h_items.begin() + n_local * DYN_SEGU, h_items.end());
                S.extra_segs.assign(h_fseg.begin() + n_local, h_fseg.end());
            }
        } else {
            // (one copy of the whole record buffer: thousands of short copies cost more than the 16 bytes per g bytes)
            const uint64_t lo = list[0] * DYN_SEGU, hi = min<uint64_t>(S.n_pos, (list[2 * (ni - 1)] + 1) * DYN_SEGU);
            CUDA_TRY(cudaMemcpyAsync(S.h_fix.data() + lo, S.d_fix + lo, (hi - lo) * sizeof(WalkRec), cudaMemcpyDeviceToHost, stream));
            CUDA_TRY(cudaStreamSynchronize(stream));
        }
        for (uint64_t k = 0; k < n_local; k++) {
            const uint64_t sg = list[2 * k];
            S.fixseg[sg] = h_fseg[k];
            S.fix_entry[sg] = list[2 * k + 1];
        }
    }
    return AMBC_OK;
}

// the chain from e, once dyn_stitch has run from it, as spans (positions relative to the span's start).  on_spec: e
// lies on the speculative chain of its segment (a walk met it there).  *raw_from = the strict stop, or untouched.
struct DynChain {
    std::vector<ChunkSpan> spans;
    std::vector<uint8_t> type;
    std::vector<uint32_t> len;
    void push(const WalkRec &r)
    {
        ChunkSpan sp; sp.pos = r.pos; sp.size = r.size; sp.pad = 0;
        spans.push_back(sp); type.push_back((uint8_t)(r.type_len >> 24)); len.push_back(r.type_len & 0xFFFFFFu);
    }
};
static int dyn_chain(const DynStitch &S, uint64_t e, bool on_spec, DynChain &C, uint64_t *raw_from)
{
    for (uint64_t sg = e / S.seglen; sg < S.n_seg && e < S.len; sg++) {
        const uint64_t s0 = sg * S.seglen, s1 = min<uint64_t>(S.len, s0 + S.seglen);
        if (e >= s1) continue;
        const WalkSeg &sp = S.h_sseg[sg];
        const WalkRec *spec = S.h_spec.data() + sg * DYN_SEGU;
        uint32_t from = 0; // first speculative record that belongs to the true chain
        bool use_spec = true;
        if (e != s0 && on_spec) {
            while (from < sp.count && spec[from].pos != e) from++;
            if (from == sp.count) return ambc_fail(AMBC_E_CUDA, "internal: meeting point not on the speculative chain");
        } else if (e != s0) {
            const WalkSeg &f = S.fixseg[sg];
            if (S.fix_entry[sg] != e) return ambc_fail(AMBC_E_CUDA, "internal: segment %llu not walked from its entry", (unsigned long long)sg);
            for (uint32_t k = 0; k < f.count; k++) C.push(S.h_fix[sg * DYN_SEGU + k]);
            if (f.merged) {
                while (from < sp.count && spec[from].pos != f.exit) from++;
                if (from == sp.count) return ambc_fail(AMBC_E_CUDA, "internal: meeting point not on the speculative chain");
            } else {
                use_spec = false;
                if (f.stop != ~0ull) { *raw_from = f.stop; break; }
                e = f.exit;
            }
        }
        on_spec = false;
        if (use_spec) {
            for (uint32_t k = from; k < sp.count; k++) C.push(spec[k]);
            if (sp.stop != ~0ull) { *raw_from = sp.stop; break; }
            e = sp.exit;
        }
    }
    return AMBC_OK;
}

// per-chunk-raw extension without a native method: raw pieces of the smallest candidate size from `from` (a multiple of
// it) up to the first piece that starts at or past `to`; `base` is subtracted from the positions
static void dyn_raw_pieces(uint64_t from, uint64_t to, uint64_t n, uint32_t cmin, uint64_t base, DynChain &C)
{
    for (uint64_t pos = from; pos < to;) {
        WalkRec r;
        r.pos = pos - base; r.size = (uint32_t)min<uint64_t>(cmin, n - pos); r.type_len = (255u << 24) | r.size;
        C.push(r);
        pos += r.size;
    }
}

// encode + frame the chosen chunks (span mode): packages only, body bytes [0, *body) of out_dev
static int dyn_encode(const uint8_t *in, uint64_t total, const DynLayout &L, uint8_t *W, const DynChain &C,
                      uint32_t method_mask, uint32_t ovh, uint32_t marker_word, uint32_t marker_bytes, void *out_dev,
                      uint64_t out_cap, uint64_t body, cudaStream_t stream)
{
    const uint64_t n_list = C.spans.size();
    if (!n_list) return AMBC_OK;
    ChunkSpan *d_spans = (ChunkSpan *)(W + L.spans);
    uint8_t *type = W + L.type;
    uint32_t *comp = (uint32_t *)(W + L.comp);
    unsigned long long *offs = (unsigned long long *)(W + L.offs);
    unsigned long long *tiles = (unsigned long long *)(W + L.tiles);
    ScanState *st = (ScanState *)(W + L.state);
    ScanState h_st;
    memset(&h_st, 0, sizeof h_st);
    h_st.first_raw = ~0ull;
    CUDA_TRY(cudaMemcpyAsync(st, &h_st, sizeof h_st, cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaMemcpyAsync(d_spans, C.spans.data(), n_list * sizeof(ChunkSpan), cudaMemcpyHostToDevice, stream));
    uint32_t maxsz = 0;
    for (uint64_t k = 0; k < n_list; k++) maxsz = max(maxsz, C.spans[k].size);
    if (maxsz > AMBC_NMAX) { // only per-chunk-raw pieces can be this large
        return ambc_fail(AMBC_E_ARG, "per-chunk-raw pieces larger than 8192 bytes are not supported");
    }
    unsigned grid = (unsigned)min<uint64_t>(n_list, 0x7fffffffull);
    int rc;
    if ((rc = launch_select_span(grid, stream, in, total, maxsz, method_mask, ovh, 0, d_spans, W + L.slots, type, comp,
                                 n_list))) return rc;
    const unsigned gt = (unsigned)((n_list + SCAN_TILE - 1) / SCAN_TILE);
    const uint32_t sflags = 1u | 2u; // every entry is a package; no END (appended by the caller)
    k_sizes<<<gt, 256, 0, stream>>>(type, comp, 0, n_list, maxsz, total, ovh, sflags, st, tiles);
    ambc_count_launch();
    k_scan_tiles<<<1, 1024, 0, stream>>>(tiles, 0, gt, 1, type, comp, n_list, maxsz, total, ovh, sflags, st, (uint8_t *)out_dev,
                                         out_cap, marker_word, marker_bytes);
    ambc_count_launch();
    k_offsets<<<gt, 256, 0, stream>>>(type, comp, 0, n_list, maxsz, total, ovh, sflags, st, tiles, offs);
    ambc_count_launch();
    size_t psmem = 32 + (((size_t)maxsz + 15) & ~(size_t)15) + 32;
    CUDA_TRY(cudaFuncSetAttribute(k_pack_span, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem));
    k_pack_span<<<grid, PACK_BLOCK, psmem, stream>>>(in, d_spans, W + L.slots, type, comp, offs, marker_word, marker_bytes,
                                                    (uint8_t *)out_dev, n_list);
    ambc_count_launch();
    CUDA_TRY(cudaGetLastError());
    // the second evaluation must agree with the trial the chain was built from
    std::vector<uint8_t> chk_t(n_list);
    std::vector<uint32_t> chk_l(n_list);
    CUDA_TRY(cudaMemcpyAsync(chk_t.data(), type, n_list, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaMemcpyAsync(chk_l.data(), comp, n_list * 4, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaMemcpyAsync(&h_st, st, sizeof h_st, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    for (uint64_t k = 0; k < n_list; k++)
        if (chk_t[k] != C.type[k] || chk_l[k] != C.len[k])
            return ambc_fail(AMBC_E_CUDA, "internal: span encode disagrees with its trial at chunk %llu", (unsigned long long)k);
    if (h_st.body_len != body) return ambc_fail(AMBC_E_CUDA, "internal: span body length mismatch");
    return AMBC_OK;
}

// usage, payload bytes and the package map of a chain (map positions shifted by `base`)
static void dyn_result(const DynChain &C, uint64_t base, ambc_compress_result *res, ambc_chunk_info *map_out, uint64_t map_cap)
{
    const uint64_t n_list = C.spans.size();
    for (uint64_t k = 0; k < n_list; k++) {
        const int t = C.type[k];
        if (t >= 1 && t <= 4) { res->usage[t]++; res->payload_bytes += C.len[k]; }
        else res->usage[0]++;
        if (map_out && k < map_cap) { map_out[k].pos = base + C.spans[k].pos; map_out[k].orig_len = C.spans[k].size; map_out[k].comp_len = C.len[k]; map_out[k].type = (uint32_t)t; }
    }
}

static uint32_t marker_word_of(const uint8_t *marker, uint32_t marker_bytes)
{
    uint32_t w = 0;
    for (uint32_t k = 0; k < marker_bytes; k++) w |= (uint32_t)marker[k] << (8 * k);
    return w;
}

extern "C" int ambc_compress_dynamic_dev(const void *in_dev, uint64_t n, const uint32_t *cands, uint32_t n_cands,
                                         uint32_t method_mask, uint32_t flags, const uint8_t *marker,
                                         uint32_t marker_bytes, void *out_dev, uint64_t out_cap, void *work_dev,
                                         uint64_t work_bytes, ambc_compress_result *res, ambc_chunk_info *map_out,
                                         uint64_t map_cap, void *stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!res || !marker || marker_bytes < 1 || marker_bytes > 4) return ambc_fail(AMBC_E_ARG, "ambc_compress_dynamic_dev: bad argument");
    if ((n && (!in_dev || !work_dev)) || !out_dev) return ambc_fail(AMBC_E_ARG, "ambc_compress_dynamic_dev: null buffer");
    DynLayout L;
    int rc = dyn_layout(n, cands, n_cands, L);
    if (rc) return rc;
    if (work_bytes < L.total) return ambc_fail(AMBC_E_CAPACITY, "ambc_compress_dynamic_dev: workspace too small");
    const uint32_t ovh = marker_bytes + 14;
    const uint32_t marker_word = marker_word_of(marker, marker_bytes);
    memset(res, 0, sizeof(*res));
    res->first_raw = -1;
    uint8_t endp[16], hdr[18];
    memcpy(endp, marker, marker_bytes);
    memset(endp + marker_bytes, 0, 12);
    uint8_t *W = (uint8_t *)work_dev;
    const bool pcr = flags & AMBC_F_PER_CHUNK_RAW;

    const bool native = (method_mask & AMBC_NATIVE_MASK) != 0;
    DynChain C;
    uint64_t raw_from = n; // raw_from < n: one raw package [raw_from, n)
    if (n && native) {
        // ---- the chain, walked on the GPU segment by segment (k_dynamic_walk), stitched from position 0 ----------
        DynStitch S;
        dyn_stitch_init(S, in_dev, n, n, cands, n_cands, method_mask, ovh, pcr, false, L, W);
        uint64_t exit, stop;
        if ((rc = dyn_spec_walk(S, stream))) return rc;
        if ((rc = dyn_stitch(S, 0, {}, &exit, &stop, stream))) return rc;
        if ((rc = dyn_chain(S, 0, false, C, &raw_from))) return rc;
    } else if (!pcr) {
        raw_from = 0; // no native method: the whole file is one raw package (:586-590)
    } else {
        dyn_raw_pieces(0, n, n, cands[n_cands - 1], 0, C);
    }
    const uint64_t n_list = C.spans.size();
    if (n_list > L.n_pos) return ambc_fail(AMBC_E_ARG, "internal: chain longer than the position table");
    uint64_t body = 0;
    for (uint64_t k = 0; k < n_list; k++) body += ovh + C.len[k];
    const uint64_t raw_len = raw_from < n ? n - raw_from : 0;
    if (raw_len > 0xFFFFFFFFull) return ambc_fail(AMBC_E_ARG, "raw package over 4 GiB cannot be framed (u32 fields)");
    const uint64_t total_body = body + (raw_len ? ovh + raw_len : 0) + marker_bytes + 12;
    if (total_body > out_cap) return ambc_fail(AMBC_E_CAPACITY, "ambc_compress_dynamic_dev: out_cap too small");

    if ((rc = dyn_encode((const uint8_t *)in_dev, n, L, W, C, method_mask, ovh, marker_word, marker_bytes, out_dev, out_cap,
                         body, stream))) return rc;
    // ---- raw tail package (if any) and END ---------------------------------------------------------
    uint8_t *o = (uint8_t *)out_dev + body;
    if (raw_len) {
        memcpy(hdr, marker, marker_bytes);
        hdr[marker_bytes] = 255; hdr[marker_bytes + 1] = 0;
        const uint32_t r32 = (uint32_t)raw_len;
        for (int r = 0; r < 3; r++) memcpy(hdr + marker_bytes + 2 + 4 * r, &r32, 4);
        CUDA_TRY(cudaMemcpyAsync(o, hdr, ovh, cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(o + ovh, (const uint8_t *)in_dev + raw_from, raw_len, cudaMemcpyDeviceToDevice, stream));
        o += ovh + raw_len;
    }
    CUDA_TRY(cudaMemcpyAsync(o, endp, marker_bytes + 12, cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));

    res->body_len = total_body;
    res->n_chunks = n_list + (raw_len ? 1 : 0);
    res->n_packages = res->n_chunks;
    res->first_raw = raw_len ? (int64_t)n_list : -1;
    dyn_result(C, 0, res, map_out, map_cap);
    if (raw_len) {
        res->usage[0]++;
        if (map_out && n_list < map_cap) { map_out[n_list].pos = raw_from; map_out[n_list].orig_len = (uint32_t)raw_len; map_out[n_list].comp_len = (uint32_t)raw_len; map_out[n_list].type = 255; }
    }
    return AMBC_OK;
}

// ---- one rank's input range of the multi-candidate mode (ambc_dyn_range_*) ------------------------------------------
// The rank walks [lo, hi) with positions relative to lo on a buffer holding [lo, min(n, hi + 8192)): the winner at p
// depends on data[p, p + 8192) and on n - p only.  lo and hi are whole segments, so the range's segments are the
// file's.  The chain enters the range at a multiple of g in [lo, lo + S), S = min(8192, cands[0]) (a non-raw package
// is at most S bytes, a per-chunk-raw piece cands[-1]): those entries are walked in segment 0 with the first round.
struct DynRangeHost {
    DynLayout L;
    DynStitch S;
    uint64_t lo, hi, n;
    uint32_t cands[32], n_cands, mask, flags, ovh;
    bool native, pcr;
    const uint8_t *buf;
    std::vector<ambc_dyn_entry> tab;
    uint64_t lo_exit, lo_stop; // the chain from lo (relative positions)
    std::vector<uint8_t> resolved; // tab[k] resolved by ambc_dyn_range_resolve: its chain was stitched past segment 0
};

static uint64_t dyn_max_entries(uint64_t g, const uint32_t *cands)
{
    return min<uint64_t>(AMBC_NMAX, cands[0]) / g;
}

extern "C" uint64_t ambc_dyn_range_workspace_bytes(uint64_t lo, uint64_t hi, uint64_t n, const uint32_t *cands,
                                                   uint32_t n_cands)
{
    DynLayout L;
    if (hi < lo || hi > n || dyn_layout(hi - lo, cands, n_cands, L)) return 0;
    if (dyn_layout(hi - lo, cands, n_cands, L, L.n_seg + dyn_max_entries(L.g, cands))) return 0;
    return L.total;
}

extern "C" int ambc_dyn_range_walk(const void *buf_dev, uint64_t buf_len, uint64_t lo, uint64_t hi, uint64_t n,
                                   const uint32_t *cands, uint32_t n_cands, uint32_t method_mask, uint32_t flags,
                                   uint32_t marker_bytes, void *work_dev, uint64_t work_bytes, ambc_dyn_range *r,
                                   ambc_dyn_entry *tab, uint32_t cap, uint32_t *n_tab, void *stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!r || !n_tab || marker_bytes < 1 || marker_bytes > 4 || hi < lo || hi > n)
        return ambc_fail(AMBC_E_ARG, "ambc_dyn_range_walk: bad argument");
    memset(r, 0, sizeof(*r));
    DynLayout L;
    int rc = dyn_layout(hi - lo, cands, n_cands, L);
    if (rc) return rc;
    const uint64_t max_e = dyn_max_entries(L.g, cands);
    if ((rc = dyn_layout(hi - lo, cands, n_cands, L, L.n_seg + max_e))) return rc;
    const uint64_t seglen = (uint64_t)DYN_SEGU * L.g;
    if ((lo % seglen && lo != n) || (hi % seglen && hi != n))
        return ambc_fail(AMBC_E_ARG, "ambc_dyn_range_walk: lo and hi must be multiples of %llu bytes or n", (unsigned long long)seglen);
    if (hi > lo && (!buf_dev || ((uintptr_t)buf_dev & 15) || buf_len < min<uint64_t>(n, hi + AMBC_NMAX) - lo))
        return ambc_fail(AMBC_E_ARG, "ambc_dyn_range_walk: the buffer must be 16-byte aligned and hold [lo, min(n, hi + 8192))");
    r->lo = lo; r->hi = hi; r->n = n; r->work_bytes = L.total;
    if (hi > lo && (!work_dev || work_bytes < L.total)) return ambc_fail(AMBC_E_CAPACITY, "ambc_dyn_range_walk: workspace too small");
    const uint64_t rlen = hi - lo;
    // the chain enters the first range at 0; any other range at one of n_e positions
    const uint64_t n_e = lo ? min<uint64_t>(max_e, (rlen + L.g - 1) / L.g) : (rlen ? 1 : 0);
    if (cap < n_e || (n_e && !tab)) return ambc_fail(AMBC_E_CAPACITY, "ambc_dyn_range_walk: entry table too small");

    DynRangeHost *H = new DynRangeHost();
    r->host = H;
    r->work_dev = work_dev;
    H->L = L; H->lo = lo; H->hi = hi; H->n = n;
    for (uint32_t i = 0; i < n_cands; i++) H->cands[i] = cands[i];
    H->n_cands = n_cands; H->mask = method_mask; H->flags = flags; H->ovh = marker_bytes + 14;
    H->native = (method_mask & AMBC_NATIVE_MASK) != 0;
    H->pcr = flags & AMBC_F_PER_CHUNK_RAW;
    H->buf = (const uint8_t *)buf_dev;
    H->tab.assign(n_e, ambc_dyn_entry());
    H->resolved.assign(n_e, 0);
    for (uint64_t k = 0; k < n_e; k++) {
        ambc_dyn_entry &t = H->tab[k];
        t.entry = lo + k * L.g; t.exit = ~0ull; t.stop = ~0ull;
    }
    if (n_e && H->native) {
        DynStitch &S = H->S;
        dyn_stitch_init(S, buf_dev, n - lo, rlen, cands, n_cands, method_mask, H->ovh, H->pcr, true, L, (uint8_t *)work_dev);
        if ((rc = dyn_spec_walk(S, stream))) return rc;
        std::vector<unsigned long long> extra;
        for (uint64_t k = 1; k < n_e; k++) { extra.push_back(0); extra.push_back(k * L.g); }
        if ((rc = dyn_stitch(S, 0, extra, &H->lo_exit, &H->lo_stop, stream))) return rc;
        for (uint64_t k = 0; k < n_e; k++) {
            ambc_dyn_entry &t = H->tab[k];
            const WalkSeg *w = k ? &S.extra_segs[k - 1] : nullptr;
            if (!k || w->merged) { // the chain from lo
                t.status = AMBC_DYN_JOIN;
                if (H->lo_stop != ~0ull) t.stop = lo + H->lo_stop;
                else t.exit = lo + H->lo_exit;
            } else if (w->stop != ~0ull) {
                t.status = AMBC_DYN_STOP; t.stop = lo + w->stop;
            } else if (w->exit >= rlen) {
                t.status = AMBC_DYN_LEAVE; t.exit = lo + w->exit;
            } else {
                t.status = AMBC_DYN_UNRESOLVED; t.exit = lo + w->exit;
            }
        }
    } else {
        // no native method: the rest of the file is raw from the entry on, or per-chunk-raw pieces of cands[-1]
        const uint64_t cmin = cands[n_cands - 1];
        for (uint64_t k = 0; k < n_e; k++) {
            ambc_dyn_entry &t = H->tab[k];
            if (!H->pcr) { t.status = AMBC_DYN_STOP; t.stop = t.entry; continue; }
            t.status = AMBC_DYN_LEAVE;
            t.exit = min<uint64_t>(n, t.entry + (hi - t.entry + cmin - 1) / cmin * cmin);
        }
    }
    for (uint64_t k = 0; k < n_e; k++) tab[k] = H->tab[k];
    *n_tab = (uint32_t)n_e;
    r->n_entries = (uint32_t)n_e;
    return AMBC_OK;
}

static int dyn_find_entry(const ambc_dyn_range *r, uint64_t entry, uint64_t *k)
{
    const DynRangeHost *H = r ? (const DynRangeHost *)r->host : nullptr;
    if (!H) return ambc_fail(AMBC_E_ARG, "ambc_dyn_range: not walked");
    for (uint64_t i = 0; i < H->tab.size(); i++)
        if (H->tab[i].entry == entry) { *k = i; return AMBC_OK; }
    return ambc_fail(AMBC_E_ARG, "ambc_dyn_range: %llu is not an entry of [%llu, %llu)", (unsigned long long)entry,
                     (unsigned long long)H->lo, (unsigned long long)H->hi);
}

extern "C" int ambc_dyn_range_resolve(ambc_dyn_range *r, uint64_t entry, ambc_dyn_entry *out, void *stream_)
{
    uint64_t k;
    int rc = dyn_find_entry(r, entry, &k);
    if (rc) return rc;
    DynRangeHost *H = (DynRangeHost *)r->host;
    ambc_dyn_entry &t = H->tab[k];
    if (t.status == AMBC_DYN_UNRESOLVED) {
        uint64_t exit, stop;
        if ((rc = dyn_stitch(H->S, t.exit - H->lo, {}, &exit, &stop, (cudaStream_t)stream_))) return rc;
        if (stop != ~0ull) { t.status = AMBC_DYN_STOP; t.stop = H->lo + stop; t.exit = ~0ull; }
        else { t.status = AMBC_DYN_LEAVE; t.exit = H->lo + exit; }
        H->resolved[k] = 1;
    }
    if (out) *out = t;
    return AMBC_OK;
}

extern "C" int ambc_dyn_range_encode(ambc_dyn_range *r, const void *buf_dev, uint64_t entry, const uint8_t *marker,
                                     uint32_t marker_bytes, void *out_dev, uint64_t out_cap, ambc_compress_result *res,
                                     ambc_chunk_info *map_out, uint64_t map_cap, uint64_t *stop, void *stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!r || !res || !stop || !marker || marker_bytes < 1 || marker_bytes > 4)
        return ambc_fail(AMBC_E_ARG, "ambc_dyn_range_encode: bad argument");
    DynRangeHost *H = (DynRangeHost *)r->host;
    if (!H) return ambc_fail(AMBC_E_ARG, "ambc_dyn_range_encode: not walked");
    if (marker_bytes + 14 != H->ovh) return ambc_fail(AMBC_E_ARG, "ambc_dyn_range_encode: marker length differs from the walk's");
    memset(res, 0, sizeof(*res));
    res->first_raw = -1;
    *stop = ~0ull;
    DynChain C;
    uint64_t raw_from = ~0ull; // relative
    if (entry < H->hi) {
        uint64_t k;
        int rc = dyn_find_entry(r, entry, &k);
        if (rc) return rc;
        const uint64_t e = entry - H->lo;
        if (!H->native) {
            if (H->pcr) dyn_raw_pieces(entry, H->hi, H->n, H->cands[H->n_cands - 1], H->lo, C);
            else raw_from = e;
        } else if (k == 0) {
            if ((rc = dyn_chain(H->S, 0, false, C, &raw_from))) return rc;
        } else {
            // the candidate's own walk in segment 0, then the chain it met, or its own stitched continuation
            const WalkSeg &w = H->S.extra_segs[k - 1];
            for (uint32_t i = 0; i < w.count; i++) C.push(H->S.extra_recs[(k - 1) * DYN_SEGU + i]);
            if (w.merged) rc = dyn_chain(H->S, w.exit, true, C, &raw_from);
            else if (w.stop != ~0ull) raw_from = w.stop;
            else if (w.exit < H->hi - H->lo) {
                if (!H->resolved[k]) return ambc_fail(AMBC_E_ARG, "ambc_dyn_range_encode: entry %llu is unresolved", (unsigned long long)entry);
                rc = dyn_chain(H->S, w.exit, false, C, &raw_from);
            }
            if (rc) return rc;
        }
    }
    const uint64_t n_list = C.spans.size();
    if (n_list > H->L.n_pos) return ambc_fail(AMBC_E_ARG, "internal: chain longer than the position table");
    uint64_t body = 0;
    for (uint64_t k = 0; k < n_list; k++) body += H->ovh + C.len[k];
    if (body > out_cap || (body && !out_dev)) return ambc_fail(AMBC_E_CAPACITY, "ambc_dyn_range_encode: out_cap too small");
    int rc = dyn_encode((const uint8_t *)buf_dev, H->n - H->lo, H->L, (uint8_t *)r->work_dev, C, H->mask, H->ovh,
                        marker_word_of(marker, marker_bytes), marker_bytes, out_dev, out_cap, body, stream);
    if (rc) return rc;
    res->body_len = body;
    res->n_chunks = res->n_packages = n_list;
    dyn_result(C, H->lo, res, map_out, map_cap);
    if (raw_from != ~0ull) *stop = H->lo + raw_from;
    return AMBC_OK;
}

extern "C" void ambc_dyn_range_free(ambc_dyn_range *r)
{
    if (!r) return;
    delete (DynRangeHost *)r->host;
    r->host = nullptr;
}
