// codec_batch.cu -- CompressionMethod plug-in entry points (compression_methods.py:7-67):
// compress() and should_use() of the four native methods over a batch of independent items.
#define AMBC_BLOCK 512 // encoder CTAs: 16 warps per chunk, 2 CTAs per SM (100 KB of shared memory each)
#include "ambc_internal.h"
#include "chunk_codec.cuh"

int ambc_deflate_encode_batch(const void *in_dev, const uint64_t *in_off_dev, uint32_t n_items, void *out_dev,
                              uint64_t out_stride, int32_t *out_len_dev, cudaStream_t stream);

extern "C" uint64_t ambc_codec_bound(int method, uint32_t n)
{
    switch (method) {
    case 1: return 2ull * n + 16;                 // one pair per byte
    case 2: return 2ull * n + 16;                 // one literal token per byte
    case 3: return 1 + 5 * 256 + 4 + 4ull * n + 16; // table + codes of at most 32 bits
    case 5: return (uint64_t)n + n / 8 + 32;        // zlib wrapper + fixed codes of at most 9 bits per byte
    default: return (uint64_t)n + 16;
    }
}

__global__ void __launch_bounds__(AMBC_BLOCK)
k_codec_encode(int method, const uint8_t *__restrict__ in, const uint64_t *__restrict__ in_off, uint32_t n_items,
               uint8_t *__restrict__ out, uint64_t out_stride, int32_t *__restrict__ out_len, int N, int pcap)
{
    extern __shared__ uint4 smem4[];
    ChunkCtx c;
    chunkctx_carve(c, (uint8_t *)smem4, N, pcap);
    for (uint32_t i = blockIdx.x; i < n_items; i += gridDim.x) {
        uint64_t a = in_off[i], b = in_off[i + 1];
        int n = (int)(b - a);
        int len = 0;
        if (n > 0) {
            chunk_load(c, in + a, n);
            if (method == 2) len = chunk_lz_encode(c);
            else if (method == 4) len = chunk_delta_encode(c);
            else {
                ChunkFeatures f;
                chunk_features(c, f);
                if (method == 1) len = chunk_rle_encode(c);
                else {
                    // K == 1 -> IndexError (:527); K == 256 -> ValueError (:382), after the tree is built
                    if (f.K <= 1) len = AMBC_CODEC_INDEX_ERROR;
                    else if (f.K == 256) len = AMBC_CODEC_VALUE_ERROR;
                    else {
                        HuffScratch hs = huff_scratch(c);
                        int bits = chunk_huff_build(c, hs, f.K);
                        len = chunk_huff_emit(c, hs, f.K, bits);
                    }
                }
            }
            __syncthreads();
            if (len > 0) copy_s2g(out + (uint64_t)i * out_stride, c.pay, min(len, pcap));
        }
        if (threadIdx.x == 0) out_len[i] = len;
        __syncthreads();
    }
}

extern "C" int ambc_codec_encode_batch(int method, const void *in_dev, const uint64_t *in_off_dev, uint32_t n_items,
                                       void *out_dev, uint64_t out_stride, int32_t *out_len_dev, void *stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (method < 1 || method > 5) return ambc_fail(AMBC_E_ARG, "ambc_codec_encode_batch: unknown method %d", method);
    if (n_items == 0) return AMBC_OK;
    if (!in_off_dev || !out_dev || !out_len_dev) return ambc_fail(AMBC_E_ARG, "null buffer");
    if (method == 5) return ambc_deflate_encode_batch(in_dev, in_off_dev, n_items, out_dev, out_stride, out_len_dev, stream);
    // item sizes are validated by the caller (<= AMBC_MAX_CODEC_CHUNK); payload capacity = stride
    const int N = AMBC_NMAX;
    uint64_t need = ambc_codec_bound(method, N);
    int pcap = (int)min<uint64_t>(out_stride, need);
    size_t smem = chunkctx_smem_bytes(N, pcap);
    CUDA_TRY(cudaFuncSetAttribute(k_codec_encode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_codec_encode<<<n_items, AMBC_BLOCK, smem, stream>>>(method, (const uint8_t *)in_dev, in_off_dev, n_items,
                                                          (uint8_t *)out_dev, out_stride, out_len_dev, N, pcap);
    ambc_count_launch();
    CUDA_TRY(cudaGetLastError());
    return AMBC_OK;
}

__global__ void __launch_bounds__(AMBC_BLOCK)
k_should_use(const uint8_t *__restrict__ in, const uint64_t *__restrict__ in_off, uint32_t n_items,
             uint8_t *__restrict__ gates, double *__restrict__ entropy, int N)
{
    extern __shared__ uint4 smem4[];
    ChunkCtx c;
    chunkctx_carve(c, (uint8_t *)smem4, N, 16);
    for (uint32_t i = blockIdx.x; i < n_items; i += gridDim.x) {
        uint64_t a = in_off[i], b = in_off[i + 1];
        int n = (int)(b - a);
        uint32_t g = 0;
        double H = 0.0;
        if (n > 0) {
            chunk_load(c, in + a, n);
            ChunkFeatures f;
            chunk_features(c, f);
            HuffScratch hs = huff_scratch(c);
            // the plug-in reports the exact Python-order sum, not the tree sum
            chunk_first_order(c, hs.firstpos, hs.order);
            H = chunk_entropy_ordered(c, f.K, hs.order);
            const int ss = min(1000, n);
            if (n >= 4 && __ddiv_rn((double)f.rep, (double)(ss - 1)) > 0.3) g |= 2u;
            if (n >= 100 && __ddiv_rn((double)f.distinct3, (double)ss) < 0.8) g |= 4u;
            if (n >= 100 && H < 7.0) g |= 8u;
            if (n >= 4 && __ddiv_rn((double)f.small, (double)(ss - 1)) > 0.5) g |= 16u;
        }
        if (threadIdx.x == 0) {
            gates[i] = (uint8_t)g;
            if (entropy) entropy[i] = H;
        }
        __syncthreads();
    }
}

extern "C" int ambc_should_use_batch(const void *in_dev, const uint64_t *in_off_dev, uint32_t n_items,
                                     uint8_t *gates_dev, double *entropy_dev, void *stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n_items == 0) return AMBC_OK;
    if (!in_off_dev || !gates_dev) return ambc_fail(AMBC_E_ARG, "null buffer");
    const int N = AMBC_NMAX;
    size_t smem = chunkctx_smem_bytes(N, 16);
    CUDA_TRY(cudaFuncSetAttribute(k_should_use, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_should_use<<<n_items, AMBC_BLOCK, smem, stream>>>((const uint8_t *)in_dev, in_off_dev, n_items, gates_dev,
                                                        entropy_dev, N);
    ambc_count_launch();
    CUDA_TRY(cudaGetLastError());
    return AMBC_OK;
}

int ambc_lz_force_buckets_codec(int on) { return lz_force_buckets_upload(on); }
