// codec_batch.cu -- CompressionMethod plug-in entry points (compression_methods.py:7-67):
// compress() and should_use() of the four native methods over a batch of independent items.  They run the
// encoders and gates of the chunk trial (select_fast.cuh): one CTA of SF_T threads per item, SfCtx<AMBC_NMAX>.
#include "ambc_internal.h"
#include "select_fast.cuh"

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

__global__ void __launch_bounds__(SF_T, 3)
k_codec_encode(int method, const uint8_t *__restrict__ in, const uint64_t *__restrict__ in_off, uint32_t n_items,
               uint8_t *__restrict__ out, uint64_t out_stride, int32_t *__restrict__ out_len)
{
    extern __shared__ uint4 smem4[];
    SfCtx<AMBC_NMAX> c;
    sf_carve<AMBC_NMAX>(c, (uint8_t *)smem4);
    for (uint32_t i = blockIdx.x; i < n_items; i += gridDim.x) {
        const uint64_t a = in_off[i];
        const int n = (int)(in_off[i + 1] - a);
        int len = 0;
        if (n > 0) {
            sf_load<AMBC_NMAX>(c, in + a, n);
            if (method == 1) {
                int pairs;
                sf_rle_features(c, &pairs); // (for the run-boundary bitmap: compress() does not ask the gate)
                len = sf_rle_emit(c);
            } else if (method == 2) {
                if (n <= 3) { // no match fits: position 0 is a literal, every later one has fewer than 3 bytes left
                    for (int p = threadIdx.x; p < n; p += SF_T) ((uint16_t *)c.pay)[p] = (uint16_t)((uint32_t)c.sd[p] << 8);
                    len = 2 * n;
                } else {
                    sf_lz_index(c);
                    len = sf_lz_parse(c, SF_ABORTED, false);
                    sf_lz_emit(c);
                }
            } else if (method == 3) {
                SfStats st;
                sf_stats(c, false, st);
                // K == 1 -> IndexError (:527); K == 256 -> ValueError (:382), after the tree is built
                if (st.K <= 1) len = AMBC_CODEC_INDEX_ERROR;
                else if (st.K == 256) len = AMBC_CODEC_VALUE_ERROR;
                else {
                    SfHuff hs = sf_huff_scratch(c);
                    const int bits = sf_huff_build(c, hs, st.K);
                    len = sf_huff_emit(c, hs, st.K, bits);
                }
            } else { // Delta (compression_methods.py:585-608)
                for (int p = threadIdx.x; p < n; p += SF_T) c.pay[p] = p ? (uint8_t)(c.sd[p] - c.sd[p - 1]) : c.sd[0];
                len = n;
            }
            __syncthreads();
            if (len > 0) copy_s2g<SF_T>(out + (uint64_t)i * out_stride, c.pay, (int)(out_stride < (uint64_t)len ? out_stride : len));
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
    // item sizes are validated by the caller (<= AMBC_MAX_CODEC_CHUNK); payloads are cut at the stride
    const int smem = SfCfg<AMBC_NMAX>::SMEM;
    CUDA_TRY(cudaFuncSetAttribute(k_codec_encode, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    k_codec_encode<<<n_items, SF_T, smem, stream>>>(method, (const uint8_t *)in_dev, in_off_dev, n_items,
                                                    (uint8_t *)out_dev, out_stride, out_len_dev);
    ambc_count_launch();
    CUDA_TRY(cudaGetLastError());
    return AMBC_OK;
}

__global__ void __launch_bounds__(SF_T, 3)
k_should_use(const uint8_t *__restrict__ in, const uint64_t *__restrict__ in_off, uint32_t n_items,
             uint8_t *__restrict__ gates, double *__restrict__ entropy)
{
    extern __shared__ uint4 smem4[];
    SfCtx<AMBC_NMAX> c;
    sf_carve<AMBC_NMAX>(c, (uint8_t *)smem4);
    for (uint32_t i = blockIdx.x; i < n_items; i += gridDim.x) {
        const uint64_t a = in_off[i];
        const int n = (int)(in_off[i + 1] - a);
        uint32_t g = 0;
        double H = 0.0;
        if (n > 0) {
            sf_load<AMBC_NMAX>(c, in + a, n);
            const int ss = min(1000, n);
            int pairs;
            if (sf_rle_features(c, &pairs)) g |= 2u; // (:154-180)
            SfStats st;
            sf_stats(c, true, st);
            if (n >= 100 && 10 * st.distinct3 < 8 * ss) g |= 4u; // distinct / ss < 0.8 (:315-343), exact as in sf_select
            // Delta (:640-667): |d[i] - d[i + 1]| < 32 at the positions range(0, n - 1, step) of the RLE gate's sample
            const int step = max(1, n / ss);
            int small = 0;
            for (int p = threadIdx.x * step; p < n - 1; p += SF_T * step) small += abs((int)c.sd[p] - (int)c.sd[p + 1]) < 32;
            small = sf_block_sum(small, c.red);
            if (n >= 4 && 2 * small > ss - 1) g |= 16u; // small / (ss - 1) > 0.5 in fp64: 0.5 is exact
            // the plug-in reports the exact Python-order entropy (DeflateCompression.should_use reads it too)
            SfHuff hs = sf_huff_scratch(c);
            sf_first_order(c, hs, st.K);
            H = sf_entropy_ordered(c, hs, st.K);
            if (n >= 100 && H < 7.0) g |= 8u; // (:551-574)
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
    const int smem = SfCfg<AMBC_NMAX>::SMEM;
    CUDA_TRY(cudaFuncSetAttribute(k_should_use, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    k_should_use<<<n_items, SF_T, smem, stream>>>((const uint8_t *)in_dev, in_off_dev, n_items, gates_dev, entropy_dev);
    ambc_count_launch();
    CUDA_TRY(cudaGetLastError());
    return AMBC_OK;
}
