// common.cuh -- shared device helpers for libambc (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#ifndef AMBC_BLOCK
#define AMBC_BLOCK 256              // threads per CTA in the chunk kernels
#endif
#define AMBC_WARPS (AMBC_BLOCK / 32)
#define AMBC_NMAX 8192              // largest chunk a native method accepts (adaptive_compressor.py:114-127)

#define FULL_MASK 0xffffffffu

// unaligned 32-bit little-endian load from shared memory (two aligned words + funnel shift)
__device__ __forceinline__ uint32_t lds_u32u(const uint8_t *s)
{
    uintptr_t a = (uintptr_t)s;
    const uint32_t *w = (const uint32_t *)(a & ~(uintptr_t)3);
    return __funnelshift_r(w[0], w[1], (uint32_t)(a & 3) * 8);
}

__device__ __forceinline__ int warp_incl_scan(int v)
{
    int lane = threadIdx.x & 31;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int t = __shfl_up_sync(FULL_MASK, v, d);
        if (lane >= d) v += t;
    }
    return v;
}

__device__ __forceinline__ int warp_sum(int v) { return __reduce_add_sync(FULL_MASK, v); } // one REDUX

// The per-warp partials of a block reduction are combined by every warp with a shuffle scan over
// lanes 0 .. AMBC_WARPS-1 (a loop over the partials costs AMBC_WARPS loads per thread).
static_assert(AMBC_WARPS <= 32, "one lane per warp partial");

// block-wide exclusive scan (AMBC_BLOCK threads).  red: >= AMBC_WARPS ints of shared memory.
// Contains two __syncthreads(); every thread of the block must call it.
__device__ __forceinline__ int block_excl_scan(int v, volatile int *red, int *total)
{
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = warp_incl_scan(v);
    __syncthreads();
    if (lane == 31) red[w] = inc;
    __syncthreads();
    int x = lane < AMBC_WARPS ? red[lane] : 0;
    int xs = warp_incl_scan(x);                          // inclusive prefix of the warp totals
    *total = __shfl_sync(FULL_MASK, xs, AMBC_WARPS - 1);
    int base = __shfl_sync(FULL_MASK, xs - x, w);        // sum of the warps before this one
    return base + inc - v;
}

// block-wide sum; two __syncthreads()
__device__ __forceinline__ int block_sum(int v, volatile int *red)
{
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    return warp_sum(lane < AMBC_WARPS ? red[lane] : 0);
}

// 16 bytes starting Q words + r bits into the eight words of two consecutive aligned 16-byte loads
template <int Q>
__device__ __forceinline__ uint4 shift16(const uint4 lo, const uint4 hi, uint32_t r)
{
    const uint32_t w[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    return make_uint4(__funnelshift_r(w[Q], w[Q + 1], r), __funnelshift_r(w[Q + 1], w[Q + 2], r),
                      __funnelshift_r(w[Q + 2], w[Q + 3], r), __funnelshift_r(w[Q + 3], w[Q + 4], r));
}

// Copy `len` bytes global -> shared.  dst is 16-byte aligned shared memory.  16-byte loads: directly when src
// is 16-byte aligned, else two aligned loads per 16 bytes, byte-shifted (package payloads start 18 bytes behind
// a package start, so this is the common case for raw pieces).  Never touches a 16-byte granule that holds no
// byte of the source range.
template <int BS = AMBC_BLOCK>
__device__ __forceinline__ void copy_g2s(uint8_t *dst, const uint8_t *__restrict__ src, int len)
{
    const int nv = len >> 4;
    uint4 *d4 = (uint4 *)dst;
    const uint32_t sh = (uint32_t)((uintptr_t)src & 15);
    if (sh == 0) {
        const uint4 *s4 = (const uint4 *)src;
        for (int i = threadIdx.x; i < nv; i += BS) d4[i] = __ldg(s4 + i);
    } else {
        const uint4 *s4 = (const uint4 *)(src - sh);
        const uint32_t r = (sh & 3) * 8;
        switch (sh >> 2) {
        case 0: for (int i = threadIdx.x; i < nv; i += BS) d4[i] = shift16<0>(__ldg(s4 + i), __ldg(s4 + i + 1), r); break;
        case 1: for (int i = threadIdx.x; i < nv; i += BS) d4[i] = shift16<1>(__ldg(s4 + i), __ldg(s4 + i + 1), r); break;
        case 2: for (int i = threadIdx.x; i < nv; i += BS) d4[i] = shift16<2>(__ldg(s4 + i), __ldg(s4 + i + 1), r); break;
        default: for (int i = threadIdx.x; i < nv; i += BS) d4[i] = shift16<3>(__ldg(s4 + i), __ldg(s4 + i + 1), r); break;
        }
    }
    for (int i = (nv << 4) + threadIdx.x; i < len; i += BS) dst[i] = __ldg(src + i);
}

// Copy `len` bytes global (any alignment) -> global (16-byte aligned), no staging: raw packages are plain bytes.
template <int BS = AMBC_BLOCK>
__device__ __forceinline__ void copy_g2g16(uint8_t *__restrict__ dst, const uint8_t *__restrict__ src, uint32_t len)
{
    const uint32_t nv = len >> 4;
    uint4 *d4 = (uint4 *)dst;
    const uint32_t sh = (uint32_t)((uintptr_t)src & 15);
    if (sh == 0) {
        const uint4 *s4 = (const uint4 *)src;
        for (uint32_t i = threadIdx.x; i < nv; i += BS) d4[i] = __ldg(s4 + i);
    } else {
        const uint4 *s4 = (const uint4 *)(src - sh);
        const uint32_t r = (sh & 3) * 8;
        switch (sh >> 2) {
        case 0: for (uint32_t i = threadIdx.x; i < nv; i += BS) d4[i] = shift16<0>(__ldg(s4 + i), __ldg(s4 + i + 1), r); break;
        case 1: for (uint32_t i = threadIdx.x; i < nv; i += BS) d4[i] = shift16<1>(__ldg(s4 + i), __ldg(s4 + i + 1), r); break;
        case 2: for (uint32_t i = threadIdx.x; i < nv; i += BS) d4[i] = shift16<2>(__ldg(s4 + i), __ldg(s4 + i + 1), r); break;
        default: for (uint32_t i = threadIdx.x; i < nv; i += BS) d4[i] = shift16<3>(__ldg(s4 + i), __ldg(s4 + i + 1), r); break;
        }
    }
    for (uint32_t i = (nv << 4) + threadIdx.x; i < len; i += BS) dst[i] = __ldg(src + i);
}

// Copy `len` bytes shared (any alignment) -> global (any alignment): byte stores up to the
// first 16-byte boundary of dst, aligned 16-byte stores fed by funnel-shifted shared loads,
// byte stores for the tail.
template <int BS = AMBC_BLOCK>
__device__ __forceinline__ void copy_s2g(uint8_t *__restrict__ dst, const uint8_t *src, int len)
{
    int head = (int)((16 - ((uintptr_t)dst & 15)) & 15);
    if (head > len) head = len;
    for (int i = threadIdx.x; i < head; i += BS) dst[i] = src[i];
    int body = (len - head) >> 4;
    uint4 *d4 = (uint4 *)(dst + head);
    const uint8_t *s = src + head;
    for (int i = threadIdx.x; i < body; i += BS) {
        const uint8_t *p = s + (i << 4);
        uint4 v;
        v.x = lds_u32u(p); v.y = lds_u32u(p + 4); v.z = lds_u32u(p + 8); v.w = lds_u32u(p + 12);
        d4[i] = v;
    }
    for (int i = head + (body << 4) + threadIdx.x; i < len; i += BS) dst[i] = src[i];
}

__device__ __forceinline__ void store_u32le(uint8_t *p, uint32_t v)
{
    p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24);
}
__device__ __forceinline__ uint32_t load_u32le(const uint8_t *p)
{
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
