// api.cu -- error reporting, bookkeeping and the host-buffer entry points of libambc.
#include "ambc_internal.h"
#include <atomic>
#include <cstdarg>
#include <mutex>
#include <vector>

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

int ambc_fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
void ambc_count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

static AmbcTiming g_timing;
AmbcTiming &ambc_timing() { return g_timing; }
void ambc_timing_mark(int idx, cudaStream_t s)
{
    if (!g_timing.on) return;
    if (!g_timing.ev[idx]) cudaEventCreate(&g_timing.ev[idx]);
    cudaEventRecord(g_timing.ev[idx], s);
}
extern "C" void ambc_enable_timing(int on) { g_timing.on = on != 0; }
extern "C" int ambc_last_timing(float *ms4)
{
    AmbcTiming &t = g_timing;
    if (!ms4) return AMBC_E_ARG;
    if (t.pending_c && t.ev[0] && t.ev[3]) {
        cudaEventSynchronize(t.ev[3]);
        cudaEventElapsedTime(&t.ms[0], t.ev[0], t.ev[1]);
        cudaEventElapsedTime(&t.ms[1], t.ev[1], t.ev[2]);
        cudaEventElapsedTime(&t.ms[2], t.ev[2], t.ev[3]);
        t.pending_c = false;
    }
    if (t.pending_d && t.ev[4] && t.ev[5]) {
        cudaEventSynchronize(t.ev[5]);
        cudaEventElapsedTime(&t.ms[3], t.ev[4], t.ev[5]);
        t.pending_d = false;
    }
    for (int i = 0; i < 4; i++) ms4[i] = t.ms[i];
    return AMBC_OK;
}

// fold of the all-gathered placement records (see include/ambc.h; mirrors distributed.fold_placement)
extern "C" int ambc_shard_place(const ambc_shard_rec *recs, uint32_t n_ranks, const uint64_t *first_byte, uint32_t chunk,
                                uint32_t marker_bytes, ambc_shard_slot *out)
{
    if (!recs || !out || !first_byte || n_ranks == 0 || chunk == 0 || marker_bytes < 1 || marker_bytes > 4)
        return ambc_fail(AMBC_E_ARG, "ambc_shard_place: bad argument");
    uint64_t offset = 0, raw_chunk = 0, raw_payload_off = 0;
    bool raw_seen = false;
    for (uint32_t r = 0; r < n_ranks; r++) {
        out[r].reserved = 0;
        if (raw_seen) { // inside the one raw package: input bytes land behind its header
            if (first_byte[r] < raw_chunk * (uint64_t)chunk) return ambc_fail(AMBC_E_ARG, "ambc_shard_place: shards out of order");
            out[r].state = AMBC_SHARD_IN_RAW_TAIL;
            out[r].offset = raw_payload_off + (first_byte[r] - raw_chunk * (uint64_t)chunk);
            continue;
        }
        out[r].offset = offset;
        offset += recs[r].packed_bytes;
        if (recs[r].first_raw >= 0) {
            if ((uint64_t)recs[r].first_raw * (uint64_t)chunk < first_byte[r]) return ambc_fail(AMBC_E_ARG, "ambc_shard_place: first_raw before the shard");
            out[r].state = AMBC_SHARD_RAW_STARTS;
            raw_seen = true;
            raw_chunk = (uint64_t)recs[r].first_raw;
            raw_payload_off = offset + marker_bytes + 14;
        } else out[r].state = AMBC_SHARD_PACKED;
    }
    return AMBC_OK;
}

extern "C" const char *ambc_last_error(void) { return g_err; }
extern "C" int ambc_version(void) { return 100; }
extern "C" uint64_t ambc_launch_count(void) { return g_launches.load(); }
extern "C" int ambc_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return ambc_fail(AMBC_E_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    return n;
}
extern "C" void *ambc_host_alloc(uint64_t bytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { ambc_fail(AMBC_E_CUDA, "cudaMallocHost failed"); return nullptr; }
    return p;
}
extern "C" void ambc_host_free(void *p) { if (p) cudaFreeHost(p); }

// ---- cached device buffers for the *_host calls (one set per device) ----------------------------
struct DevBuf {
    void *p = nullptr;
    uint64_t cap = 0;
    int ensure(uint64_t bytes)
    {
        if (bytes <= cap) return AMBC_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        uint64_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { p = nullptr; return ambc_fail(AMBC_E_CUDA, "cudaMalloc(%llu): %s", (unsigned long long)want, cudaGetErrorString(e)); }
        cap = want;
        return AMBC_OK;
    }
};
#define AMBC_MAX_PIECES 64
struct HostCtx {
    DevBuf in, out, work, table, status;
    cudaStream_t stream = nullptr, copy = nullptr, d2h = nullptr, aux = nullptr;
    cudaEvent_t piece_ev[AMBC_MAX_PIECES] = {};
    cudaEvent_t ring_ev[4] = {};
    cudaEvent_t done_ev[AMBC_MAX_PIECES] = {};
    cudaEvent_t sel_ev[AMBC_MAX_PIECES] = {};
    void *states = nullptr; // pinned scan states, one per piece
    bool ring_used[4] = {false, false, false, false};
    void *table_host = nullptr; // pinned ring of table pieces (ambc_decompress_host)
};
int ambc_index_vector(const uint8_t *body, uint64_t body_len, const uint8_t *marker, uint32_t mb, uint64_t orig_size,
                      uint32_t known_mask, std::vector<ambc_pkg> &v, uint64_t *n_entries, uint64_t *out_bytes);
int ambc_compress_dev_impl(const void *in_dev, uint64_t n, uint32_t chunk, uint32_t method_mask, uint32_t flags,
                           const uint8_t *marker, uint32_t marker_bytes, void *out_dev, uint64_t out_cap,
                           void *work_dev, uint64_t work_bytes, ambc_compress_result *res, cudaStream_t stream,
                           const cudaEvent_t *piece_ready, const uint64_t *piece_start, uint32_t n_pieces,
                           const AmbcPieceOut *po);
static std::mutex g_mu;
static HostCtx g_ctx[16];

static int host_ctx(HostCtx **out)
{
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return ambc_fail(AMBC_E_CUDA, "cudaGetDevice: %s (no CUDA device? libambc has no CPU fallback)", cudaGetErrorString(e));
    if (dev < 0 || dev >= 16) return ambc_fail(AMBC_E_ARG, "device index out of range");
    HostCtx *c = &g_ctx[dev];
    if (!c->stream) {
        e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) return ambc_fail(AMBC_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
        e = cudaStreamCreateWithFlags(&c->copy, cudaStreamNonBlocking);
        if (e != cudaSuccess) return ambc_fail(AMBC_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
        e = cudaStreamCreateWithFlags(&c->d2h, cudaStreamNonBlocking);
        if (e != cudaSuccess) return ambc_fail(AMBC_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
        e = cudaStreamCreateWithFlags(&c->aux, cudaStreamNonBlocking);
        if (e != cudaSuccess) return ambc_fail(AMBC_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
        for (int i = 0; i < AMBC_MAX_PIECES; i++) cudaEventCreateWithFlags(&c->sel_ev[i], cudaEventDisableTiming);
        for (int i = 0; i < AMBC_MAX_PIECES; i++) cudaEventCreateWithFlags(&c->piece_ev[i], cudaEventDisableTiming);
        for (int i = 0; i < 4; i++) cudaEventCreateWithFlags(&c->ring_ev[i], cudaEventDisableTiming);
        for (int i = 0; i < AMBC_MAX_PIECES; i++) cudaEventCreateWithFlags(&c->done_ev[i], cudaEventDisableTiming);
    }
    *out = c;
    return AMBC_OK;
}

extern "C" int ambc_compress_host(const void *in_host, uint64_t n, uint32_t chunk, uint32_t method_mask,
                                  uint32_t flags, const uint8_t *marker, uint32_t marker_bytes, void *out_host,
                                  uint64_t out_cap, uint8_t *map_type, uint32_t *map_comp, ambc_compress_result *res)
{
    std::lock_guard<std::mutex> lk(g_mu);
    HostCtx *c;
    int rc = host_ctx(&c);
    if (rc) return rc;
    if (!res || chunk == 0) return ambc_fail(AMBC_E_ARG, "ambc_compress_host: bad argument");
    uint64_t bound = ambc_compress_bound(n, chunk, marker_bytes);
    uint64_t wbytes = ambc_compress_workspace_bytes(n, chunk);
    if ((rc = c->in.ensure(n + 64))) return rc;
    if ((rc = c->out.ensure(bound))) return rc;
    if ((rc = c->work.ensure(wbytes))) return rc;
    // upload in pieces on a second stream; select / scan / pack of piece k start as soon as piece k is
    // resident, and finished body bytes are downloaded while later pieces compute.  Pieces are whole scan
    // tiles (2048 chunks); they ramp 8 -> 16 -> 32 -> 64 MiB at the front (k_select starts early) and back
    // down at the end (little left to pack and download after the last k_select)
    const uint64_t n_chunks = (n + chunk - 1) / chunk;
    const uint64_t tile_bytes = 2048ull * chunk, n_tiles = (n_chunks + 2047) / 2048;
    uint64_t unit = max<uint64_t>(1, (8ull << 20) / tile_bytes), big = max<uint64_t>(unit, (64ull << 20) / tile_bytes);
    std::vector<uint64_t> sizes; // in tiles
    for (;;) {
        sizes.clear();
        std::vector<uint64_t> ramp;
        for (uint64_t r = unit; r < big; r *= 2) ramp.push_back(r);
        uint64_t ramp_sum = 0;
        for (uint64_t r : ramp) ramp_sum += r;
        if (n_tiles >= 2 * ramp_sum + big) {
            uint64_t mid = n_tiles - 2 * ramp_sum;
            sizes = ramp;
            for (; mid >= 2 * big; mid -= big) sizes.push_back(big);
            sizes.push_back(mid);
            for (size_t r = ramp.size(); r-- > 0;) sizes.push_back(ramp[r]);
        } else {
            for (uint64_t t = 0; t < n_tiles; t += big) sizes.push_back(min<uint64_t>(big, n_tiles - t));
        }
        if (sizes.size() <= AMBC_MAX_PIECES) break;
        big *= 2; // (very large inputs: fewer, larger pieces)
    }
    const uint64_t n_pieces = sizes.size();
    uint64_t piece_start[AMBC_MAX_PIECES + 1];
    piece_start[0] = 0;
    for (uint64_t k = 0; k < n_pieces; k++) piece_start[k + 1] = piece_start[k] + sizes[k] * 2048;
    if (!c->states) {
        if (cudaMallocHost(&c->states, AMBC_MAX_PIECES * ambc_scan_state_bytes()) != cudaSuccess)
            return ambc_fail(AMBC_E_CUDA, "cudaMallocHost failed");
    }
    AmbcPieceOut po;
    po.out_host = out_host; po.out_cap = out_cap; po.states = c->states; po.done = c->done_ev; po.d2h = c->d2h;
    po.aux = c->aux; po.sel = c->sel_ev;
    if (n_pieces > 1) {
        for (uint64_t k = 0; k < n_pieces; k++) {
            uint64_t b0 = piece_start[k] * chunk, b1 = min<uint64_t>(n, piece_start[k + 1] * chunk);
            CUDA_TRY(cudaMemcpyAsync((uint8_t *)c->in.p + b0, (const uint8_t *)in_host + b0, b1 - b0, cudaMemcpyHostToDevice, c->copy));
            CUDA_TRY(cudaEventRecord(c->piece_ev[k], c->copy));
        }
        rc = ambc_compress_dev_impl(c->in.p, n, chunk, method_mask, flags, marker, marker_bytes, c->out.p, bound, c->work.p,
                                    c->work.cap, res, c->stream, c->piece_ev, piece_start, (uint32_t)n_pieces, &po);
    } else {
        if (n) CUDA_TRY(cudaMemcpyAsync(c->in.p, in_host, n, cudaMemcpyHostToDevice, c->stream));
        rc = ambc_compress_dev_impl(c->in.p, n, chunk, method_mask, flags, marker, marker_bytes, c->out.p, bound, c->work.p,
                                    c->work.cap, res, c->stream, nullptr, nullptr, 0, &po);
    }
    if (rc) { cudaStreamSynchronize(c->copy); return rc; }
    if (map_type && res->n_chunks)
        CUDA_TRY(cudaMemcpyAsync(map_type, (uint8_t *)c->work.p + res->map_type_off, res->n_chunks,
                                 cudaMemcpyDeviceToHost, c->stream));
    if (map_comp && res->n_chunks)
        CUDA_TRY(cudaMemcpyAsync(map_comp, (uint8_t *)c->work.p + res->map_comp_off, res->n_chunks * 4,
                                 cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return AMBC_OK;
}

int ambc_index_stream(const uint8_t *body, uint64_t body_len, const uint8_t *marker, uint32_t mb, uint64_t orig_size,
                      uint32_t known_mask, void (*sink)(void *, const ambc_pkg &), void *user, uint64_t *n_entries,
                      uint64_t *out_bytes);
int ambc_decode_launch(const void *body_dev, const ambc_pkg *table_dev, uint64_t n_entries, void *out_dev,
                       uint32_t *status_dev, cudaStream_t stream, uint32_t known_mask);

// state of the piece-wise decode that runs while the host walks the package chain
struct DecPipe {
    HostCtx *c;
    const uint8_t *body_host;
    uint8_t *out_host;
    uint64_t body_len, uploaded = 0; // body bytes whose upload has been queued on the copy stream
    uint64_t filled = 0, flushed_entries = 0;
    uint64_t piece_entries = 2048; // ramps up to DEC_PIECE_ENTRIES so the first download starts early
    uint32_t known_mask = 0;       // packages of types 6 / 7 are decoded when their bits are set
    int rc = AMBC_OK;
    int ev = 0, ring = 0, up = 0;
};
#define DEC_PIECE_ENTRIES 16384
#define DEC_RING 4                     // table pieces in flight (pinned host + device copies)
#define DEC_BODY_PIECE (16ull << 20)   // body upload granule
#define DEC_BODY_AHEAD (32ull << 20)   // body bytes queued ahead of the walk

// queue body uploads until at least `upto` bytes (capped at the body) are on their way
static void decpipe_upload(DecPipe &d, uint64_t upto)
{
    HostCtx *c = d.c;
    if (upto > d.body_len) upto = d.body_len;
    while (d.uploaded < upto && !d.rc) {
        uint64_t nb = min<uint64_t>(DEC_BODY_PIECE, d.body_len - d.uploaded);
        cudaError_t e = cudaMemcpyAsync((uint8_t *)c->in.p + d.uploaded, d.body_host + d.uploaded, nb,
                                        cudaMemcpyHostToDevice, c->copy);
        if (e != cudaSuccess) { d.rc = ambc_fail(AMBC_E_CUDA, "body upload: %s", cudaGetErrorString(e)); return; }
        d.uploaded += nb;
    }
}

static void decpipe_flush(DecPipe &d)
{
    if (d.rc || d.filled == 0) return;
    HostCtx *c = d.c;
    // ring slot r (pinned host piece + its device copy) is free again once the kernels of its previous piece ran
    const ambc_pkg *src = (const ambc_pkg *)c->table_host + (uint64_t)d.ring * DEC_PIECE_ENTRIES;
    ambc_pkg *tab_dev = (ambc_pkg *)c->table.p + (uint64_t)d.ring * DEC_PIECE_ENTRIES;
    // copy stream, in order: the body bytes these packages read, their table piece, then some body ahead
    const uint64_t need = src[d.filled - 1].src_off + src[d.filled - 1].comp_len;
    decpipe_upload(d, need);
    if (d.rc) return;
    cudaError_t e = cudaMemcpyAsync(tab_dev, src, d.filled * sizeof(ambc_pkg), cudaMemcpyHostToDevice, c->copy);
    if (e != cudaSuccess) { d.rc = ambc_fail(AMBC_E_CUDA, "table upload: %s", cudaGetErrorString(e)); return; }
    cudaEvent_t up = c->done_ev[d.up];
    d.up = (d.up + 1) % AMBC_MAX_PIECES;
    cudaEventRecord(up, c->copy);
    cudaStreamWaitEvent(c->stream, up, 0);
    decpipe_upload(d, need + DEC_BODY_AHEAD);
    if (d.rc) return;
    d.rc = ambc_decode_launch(c->in.p, tab_dev, d.filled, c->out.p, (uint32_t *)c->status.p, c->stream, d.known_mask);
    if (d.rc) return;
    // results of this piece go home on the download stream while the walk and the next kernels continue
    const uint64_t d0 = src[0].dst_off, d1 = src[d.filled - 1].dst_off + src[d.filled - 1].out_len;
    cudaEvent_t ev = c->piece_ev[d.ev];
    d.ev = (d.ev + 1) % AMBC_MAX_PIECES;
    cudaEventRecord(ev, c->stream);
    cudaEventRecord(c->ring_ev[d.ring], c->stream);
    c->ring_used[d.ring] = true;
    d.ring = (d.ring + 1) % DEC_RING;
    cudaStreamWaitEvent(c->d2h, ev, 0);
    e = cudaMemcpyAsync(d.out_host + d0, (uint8_t *)c->out.p + d0, d1 - d0, cudaMemcpyDeviceToHost, c->d2h);
    if (e != cudaSuccess) { d.rc = ambc_fail(AMBC_E_CUDA, "result download: %s", cudaGetErrorString(e)); return; }
    d.flushed_entries += d.filled;
    d.filled = 0;
    if (d.piece_entries < DEC_PIECE_ENTRIES) d.piece_entries *= 2;
    // the next piece is written into the next ring slot: wait until the GPU is done with it
    if (c->ring_used[d.ring]) cudaEventSynchronize(c->ring_ev[d.ring]);
}

static void decpipe_sink(void *user, const ambc_pkg &e)
{
    DecPipe &d = *(DecPipe *)user;
    if (d.rc) return;
    ((ambc_pkg *)d.c->table_host)[(uint64_t)d.ring * DEC_PIECE_ENTRIES + d.filled++] = e;
    if (d.filled == d.piece_entries) decpipe_flush(d);
}


extern "C" int ambc_decompress_host(const void *body_host, uint64_t body_len, const uint8_t *marker,
                                    uint32_t marker_bytes, uint32_t known_mask, void *out_host, uint64_t orig_size,
                                    uint32_t *status)
{
    std::lock_guard<std::mutex> lk(g_mu);
    HostCtx *c;
    int rc = host_ctx(&c);
    if (rc) return rc;
    if (!marker || marker_bytes < 1 || marker_bytes > 4) return ambc_fail(AMBC_E_ARG, "ambc_decompress_host: bad marker");
    uint64_t ne = 0, covered = 0;
    // the body upload (in DEC_BODY_PIECE granules, a little ahead of the walk), the host walk of the package
    // chain, the decode kernels and the download of finished pieces all overlap: the walk hands
    // DEC_PIECE_ENTRIES packages at a time to the GPU, which needs only the body bytes up to their end
    if ((rc = c->in.ensure(body_len + 64))) return rc;
    if ((rc = c->out.ensure(orig_size + 64))) return rc;
    if ((rc = c->status.ensure(64))) return rc;
    if ((rc = c->table.ensure((uint64_t)DEC_RING * DEC_PIECE_ENTRIES * sizeof(ambc_pkg) + 64))) return rc;
    for (int i = 0; i < DEC_RING; i++) c->ring_used[i] = false;
    if (!c->table_host &&
        cudaMallocHost(&c->table_host, (uint64_t)DEC_RING * DEC_PIECE_ENTRIES * sizeof(ambc_pkg)) != cudaSuccess)
        return ambc_fail(AMBC_E_CUDA, "cudaMallocHost failed");
    CUDA_TRY(cudaMemsetAsync(c->status.p, 0, 8, c->stream));
    DecPipe d;
    d.c = c; d.body_host = (const uint8_t *)body_host; d.out_host = (uint8_t *)out_host; d.body_len = body_len;
    d.known_mask = known_mask;
    decpipe_upload(d, DEC_BODY_AHEAD);
    if (d.rc) return d.rc;
    rc = ambc_index_stream((const uint8_t *)body_host, body_len, marker, marker_bytes, orig_size, known_mask,
                           decpipe_sink, &d, &ne, &covered);
    if (!rc) { decpipe_flush(d); rc = d.rc; }
    if (rc) { cudaStreamSynchronize(c->copy); cudaStreamSynchronize(c->stream); cudaStreamSynchronize(c->d2h); return rc; }
    if (covered < orig_size) { // zero pad (adaptive_compressor.py:447-449)
        memset((uint8_t *)out_host + covered, 0, orig_size - covered);
    }
    uint32_t st[2] = {0, 0};
    CUDA_TRY(cudaMemcpyAsync(st, c->status.p, 8, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->copy));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->d2h));
    if (status) { status[0] = st[0]; status[1] = st[1]; }
    return AMBC_OK;
}
