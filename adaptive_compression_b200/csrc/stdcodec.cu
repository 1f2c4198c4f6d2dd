// stdcodec.cu -- decode kernels of method ids 6 (BZip2Compression, bzip2.cuh) and 7 (LZMACompression, xz.cuh), for
// packages in a body (the table of ambc_index_host / ambc_index_dev) and for the plug-in batch call.
//   LZMA:  one package per one-warp CTA.  Lane 0 runs the range decoder; the probability model (at most 28268 bytes
//          for lc + lp = 4) is in shared memory; the package's own output is the dictionary, so no global scratch.
//   bzip2: one package per one-warp CTA.  Lane 0 decodes (Huffman, inverse MTF, inverse BWT, run-of-4); the tables
//          (about 29 KiB) are in shared memory, the block (4 bytes per block byte: symbol and T vector) in a global
//          scratch slot of BZ2_MAX_BLOCK words per resident CTA.
// The other lanes zero-pad the output.  Where the stock library raises, the output is original_length zero bytes.
#include "ambc_internal.h"
#include "common.cuh"
#include "bzip2.cuh"
#include "xz.cuh"

#define STD_LZMA_CTAS (148 * 8) // 8 x 28 KiB of probabilities fit in an SM's shared memory
#define STD_BZ2_CTAS (148 * 2)  // each holds a 3.6 MB scratch slot

// where a decoder's work comes from: the package table of a body, or the items of a batch call
struct StdJob {
    // container
    const uint8_t *body;
    const ambc_pkg *table;
    uint64_t n_entries;
    uint8_t *out;
    uint32_t *status;
    // batch
    const uint8_t *in;
    const uint64_t *in_off;
    const uint32_t *orig_len;
    uint64_t out_stride;
    int32_t *out_len;
};

// the CTA's next package of type `type`: *i advances through entries blockIdx.x + k * gridDim.x, 32 at a time
__device__ bool std_next(const StdJob &j, uint32_t type, uint64_t &k0, uint32_t &todo, uint64_t *i)
{
    const int lane = threadIdx.x & 31;
    const uint64_t n = j.n_entries;
    while (!todo) {
        if (blockIdx.x + k0 * gridDim.x >= n) return false;
        const uint64_t mine = blockIdx.x + (k0 + lane) * (uint64_t)gridDim.x;
        const bool want = mine < n && (!j.table || j.table[mine].type == type);
        todo = __ballot_sync(FULL_MASK, want);
        if (!todo) k0 += 32;
    }
    const int b = __ffs(todo) - 1;
    todo &= todo - 1;
    *i = blockIdx.x + (k0 + b) * (uint64_t)gridDim.x;
    if (!todo) k0 += 32;
    return true;
}

// one package or item: lane 0 decodes, then the warp pads / zero-fills and reports
template <class Decode>
__device__ void std_item(const StdJob &j, uint64_t i, Decode dec)
{
    const int lane = threadIdx.x & 31;
    const uint8_t *src;
    uint8_t *dst;
    uint64_t comp, want, bufsz;
    uint32_t orig;
    if (j.table) {
        const ambc_pkg e = j.table[i];
        src = j.body + e.src_off; comp = e.comp_len; orig = e.orig_len;
        dst = j.out + e.dst_off; want = e.out_len; bufsz = e.out_len; // no room behind a package
    } else {
        src = j.in + j.in_off[i]; comp = j.in_off[i + 1] - j.in_off[i]; orig = j.orig_len[i];
        dst = j.out + i * j.out_stride; want = orig < j.out_stride ? orig : j.out_stride; bufsz = j.out_stride;
    }
    long got = 0;
    if (comp > 0 && lane == 0) got = dec(src, (long)comp, dst, (long)want, (long)bufsz);
    got = __shfl_sync(FULL_MASK, (long long)got, 0);
    // got: total decoded bytes, -1 where the stock library raises, -2 output stopped at bufsz
    const uint64_t good = got < 0 ? (got == -2 ? want : 0) : ((uint64_t)got < want ? (uint64_t)got : want);
    __syncwarp();
    if (comp > 0)
        for (uint64_t k = good + lane; k < want; k += 32) dst[k] = 0;
    if (lane == 0) {
        if (j.table) {
            if (got == -1 && j.status) atomicAdd(&j.status[0], 1u);
        } else {
            // an empty payload decodes to b''; a stream that needs more room than the stride is reported
            j.out_len[i] = comp == 0 ? 0 : (got == -2 ? AMBC_E_CAPACITY : (int32_t)orig);
        }
    }
    __syncwarp();
}

__global__ void __launch_bounds__(32) k_lzma_decode(StdJob j)
{
    extern __shared__ uint4 smem4[];
    uint16_t *probs = (uint16_t *)smem4;
    uint64_t k0 = 0, i;
    uint32_t todo = 0;
    while (std_next(j, 7, k0, todo, &i))
        std_item(j, i, [&](const uint8_t *src, long comp, uint8_t *dst, long want, long bufsz) -> long {
            (void)want;
            return xz_decompress(src, comp, dst, bufsz, probs);
        });
}

__global__ void __launch_bounds__(32) k_bz2_decode(StdJob j, uint32_t *tt_all)
{
    extern __shared__ uint4 smem4[];
    Bz2Work *w = (Bz2Work *)smem4;
    uint32_t *tt = tt_all + (uint64_t)blockIdx.x * BZ2_MAX_BLOCK;
    uint64_t k0 = 0, i;
    uint32_t todo = 0;
    while (std_next(j, 6, k0, todo, &i))
        std_item(j, i, [&](const uint8_t *src, long comp, uint8_t *dst, long want, long bufsz) -> long {
            (void)bufsz;
            return bz2_decompress(src, comp, dst, want, w, tt);
        });
}

// bzip2 scratch, one set of slots per device, allocated on first use and kept
static void *g_bz2_tt[16];

static int std_launch(int method, const StdJob &j, uint64_t n, cudaStream_t stream)
{
    if (n == 0) return AMBC_OK;
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 16) return ambc_fail(AMBC_E_ARG, "device index out of range");
    static bool attr_done[16] = {};
    if (!attr_done[dev]) {
        CUDA_TRY(cudaFuncSetAttribute(k_lzma_decode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(LZMA_PROBS_MAX * 2)));
        CUDA_TRY(cudaFuncSetAttribute(k_bz2_decode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Bz2Work)));
        attr_done[dev] = true;
    }
    if (method == 7) {
        const unsigned grid = (unsigned)min<uint64_t>(n, STD_LZMA_CTAS);
        k_lzma_decode<<<grid, 32, LZMA_PROBS_MAX * 2, stream>>>(j);
    } else {
        if (!g_bz2_tt[dev]) {
            cudaError_t e = cudaMalloc(&g_bz2_tt[dev], (size_t)STD_BZ2_CTAS * BZ2_MAX_BLOCK * sizeof(uint32_t));
            if (e != cudaSuccess) { g_bz2_tt[dev] = nullptr; return ambc_fail(AMBC_E_CUDA, "bzip2 scratch: %s", cudaGetErrorString(e)); }
        }
        const unsigned grid = (unsigned)min<uint64_t>(n, STD_BZ2_CTAS);
        k_bz2_decode<<<grid, 32, sizeof(Bz2Work), stream>>>(j, (uint32_t *)g_bz2_tt[dev]);
    }
    ambc_count_launch();
    CUDA_TRY(cudaGetLastError());
    return AMBC_OK;
}

// packages of type 6 / 7 in table[0 .. n_entries) (the bits of known_mask say which of the two to look for)
int ambc_stdcodec_decode_table(const void *body_dev, const ambc_pkg *table_dev, uint64_t n_entries, void *out_dev,
                               uint32_t *status_dev, uint32_t known_mask, cudaStream_t stream)
{
    StdJob j = {};
    j.body = (const uint8_t *)body_dev; j.table = table_dev; j.n_entries = n_entries;
    j.out = (uint8_t *)out_dev; j.status = status_dev;
    int rc;
    if ((known_mask >> 7) & 1u)
        if ((rc = std_launch(7, j, n_entries, stream))) return rc;
    if ((known_mask >> 6) & 1u)
        if ((rc = std_launch(6, j, n_entries, stream))) return rc;
    return AMBC_OK;
}

int ambc_stdcodec_decode_batch(int method, const void *in_dev, const uint64_t *in_off_dev, const uint32_t *orig_len_dev,
                               uint32_t n_items, void *out_dev, uint64_t out_stride, int32_t *out_len_dev, cudaStream_t stream)
{
    StdJob j = {};
    j.in = (const uint8_t *)in_dev; j.in_off = in_off_dev; j.orig_len = orig_len_dev; j.n_entries = n_items;
    j.out = (uint8_t *)out_dev; j.out_stride = out_stride; j.out_len = out_len_dev;
    return std_launch(method, j, n_items, stream);
}
