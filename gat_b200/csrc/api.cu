// api.cu -- the C ABI of libgat_b200.so (include/gat_b200.h): contexts, staging, batching.
//
// Host code here only moves data and sequences kernel launches; every interval computation of the
// hot path runs in the CUDA kernels of place.cu / count.cu.  There is no CPU fallback: if CUDA is
// unavailable every compute entry point returns GATB_ERR_CUDA.
#include "../../include/gat_b200.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <memory>
#include <string>
#include <vector>

#include "count.cuh"
#include "place.cuh"

using namespace gatb;

// ---------------------------------------------------------------------------------------------------
struct gatb_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaStream_t upload_stream = nullptr;   // gatb_annotations_create_async: copies (+ a rebuild), off the compute stream
    cudaStream_t build_stream = nullptr;    // index build kernels, chunk by chunk behind the copies
    cudaStream_t copy_stream = nullptr;     // gatb_run with host outputs: device-to-host copies of batch i overlap batch i+1
    cudaEvent_t ev_counted[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
    uint32_t *err_slots = nullptr;          // pinned words of pending asynchronous creates: 4 per set (validation, -, entries needed lo/hi)
    uint8_t *small_stage = nullptr;         // pinned: 16 KB per pending set for its small host-built tables (a copy from
                                            // pageable memory makes cudaMemcpyAsync wait for other work of the context)
    std::vector<int> err_free;
    std::string err;
    uint64_t launches = 0;
    uint32_t batch = 0;                 // 0 = default
    int sm_count = 148;
    size_t smem_optin = 0;
    // tunables (env overrides, for profiling)
    int count_threads = 1024;
    uint32_t schunk_max = 0;            // samples per count CTA; 0: whatever shared memory allows
    uint32_t kgrp_max = 0;              // keys per item table; 0: whatever fits
    struct BatchScratch *scratch = nullptr;
    struct BlockCache *blocks = nullptr;
    // output routes of gatb_run (gatb_set_output_routes): integer counts delivered to several destinations,
    // possibly peer GPUs, by the counting kernel's epilogue
    std::vector<gatb_route> routes;
    bool stats_stream = true;           // uint32 column statistics as TMA-streamed passes (GATB_STATS_STREAM=0: the column-tiled kernels)
    bool route_copy = true;             // routes are served by copy engines from a staging slab (false: by the kernel's stores)
    bool trace = false;                 // GATB_TRACE=1: host-side phase times of gatb_run on stderr
    // optional per-kernel timing (bench.py roofline): CUDA events around every launch
    bool profiling = false;
    struct Span { int cls; cudaEvent_t a, b; };
    std::vector<Span> spans;
};

constexpr size_t SMALL_STAGE_BYTES = 16384;
enum { PROF_PLACE = 0, PROF_MERGE = 1, PROF_COUNT = 2, PROF_OTHER = 3, PROF_NCLS = 4 };

struct ProfScope {
    gatb_ctx *ctx; int cls; cudaStream_t st; cudaEvent_t a = nullptr, b = nullptr;
    ProfScope(gatb_ctx *c, int k, cudaStream_t stream = nullptr) : ctx(c), cls(k), st(stream ? stream : c->stream)
    {
        ctx->launches++;
        if (!ctx->profiling) return;
        cudaEventCreate(&a); cudaEventCreate(&b);
        cudaEventRecord(a, st);
    }
    ~ProfScope()
    {
        if (!a) return;
        cudaEventRecord(b, st);
        ctx->spans.push_back({cls, a, b});
    }
};

// Recycled device blocks for the large index arrays of annotation sets (entries, exact intervals, previous ends, bin
// offsets / records: ~2 GB per 1000-track set).  A caller that builds a set per call -- bench.py's e2e leg, gat.run per
// key tuple -- would otherwise return 2 GB to the stream-ordered pool and ask for it again every time; under multi-process
// peer mappings the pool was seen to go back to the driver for part of it every step (5-45 ms of host time).  Blocks are
// handed out and taken back in upload-stream order (gatb_annotations_destroy makes that stream wait for the compute
// stream first), so a recycled block is never written while its previous user still reads it.
struct BlockCache {
    struct Block { void *p; size_t bytes; };
    std::vector<Block> free_blocks;
    size_t cached = 0;
    static constexpr size_t LIMIT = 12ull << 30;
    void *take(size_t bytes, size_t *got)
    {
        int best = -1;
        for (size_t i = 0; i < free_blocks.size(); i++)
            if (free_blocks[i].bytes >= bytes && free_blocks[i].bytes <= bytes + bytes / 2 + (1u << 20) &&
                (best < 0 || free_blocks[i].bytes < free_blocks[(size_t)best].bytes)) best = (int)i;
        if (best < 0) return nullptr;
        void *p = free_blocks[(size_t)best].p;
        *got = free_blocks[(size_t)best].bytes;
        cached -= *got;
        free_blocks.erase(free_blocks.begin() + best);
        return p;
    }
    bool give(void *p, size_t bytes)
    {
        if (bytes < (8u << 20) || cached + bytes > LIMIT) return false;
        free_blocks.push_back({p, bytes});
        cached += bytes;
        return true;
    }
    void drop(cudaStream_t st)
    {
        for (auto &b : free_blocks) if (cudaFreeAsync(b.p, st) != cudaSuccess) { cudaGetLastError(); cudaFree(b.p); }
        free_blocks.clear();
        cached = 0;
    }
};

static std::string g_create_err;

static int fail(gatb_ctx *ctx, int code, const std::string &msg)
{
    if (ctx) ctx->err = msg; else g_create_err = msg;
    return code;
}

#define CU(ctx, call)                                                                             \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess)                                                                   \
            return fail(ctx, GATB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
    } while (0)

// Device buffers come from the stream-ordered allocator (cudaMallocAsync on the context's stream, pool
// release threshold unlimited): creating and destroying samplers / annotation sets per call re-uses
// pooled memory instead of paying cudaMalloc/cudaFree (which synchronise the device) every time.
static thread_local cudaStream_t tl_stream = nullptr;

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    cudaStream_t st = nullptr;
    BlockCache *cache = nullptr;         // alloc_cached: where the block goes back to
    size_t block_bytes = 0;
    ~DevBuf() { release(); }
    void release()
    {
        if (p && cache && cache->give(p, block_bytes)) p = nullptr;
        if (p && cudaFreeAsync(p, st) != cudaSuccess) { cudaGetLastError(); cudaFree(p); }
        p = nullptr; n = 0; cache = nullptr;
    }
    cudaError_t alloc(size_t count)
    {
        release();
        n = count;
        st = tl_stream;
        if (count == 0) return cudaSuccess;
        return cudaMallocAsync((void **)&p, count * sizeof(T), st);
    }
    // a block from the context's recycling cache (large index arrays, see BlockCache), else a fresh one
    cudaError_t alloc_cached(BlockCache *bc, size_t count)
    {
        release();
        n = count;
        st = tl_stream;
        if (count == 0) return cudaSuccess;
        block_bytes = count * sizeof(T);
        cache = bc;
        if (void *q = bc->take(block_bytes, &block_bytes)) { p = (T *)q; return cudaSuccess; }
        return cudaMallocAsync((void **)&p, block_bytes, st);
    }
    cudaError_t ensure(size_t count) { return count <= n ? cudaSuccess : alloc(count); }
    cudaError_t upload(const T *h, size_t count, cudaStream_t stream)
    {
        cudaError_t e = alloc(count);
        if (e != cudaSuccess || count == 0) return e;
        return cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, stream);
    }
};

// Batch buffers of the sampling loop, owned by the context and only ever grown: samplers created and
// destroyed per call (one per track in gat.run) re-use them instead of allocating hundreds of MB each.
// Calls on a context are serialised by the caller and every entry point that uses the buffers returns
// with the stream drained, so sharing them between samplers is safe.
struct PlaceBufs {                        // one batch of placed samples
    DevBuf<uint64_t> unit_buf, placed;
    DevBuf<uint32_t> unit_n, placed_n;
    DevBuf<uint8_t> status;
};
struct BatchScratch {
    PlaceBufs pb;
    DevBuf<uint32_t> out_tmp[2];          // host-output runs: two staging slabs, so that the copy of batch i
    DevBuf<double> out_tmp_f[2];          // to the host overlaps the kernels of batch i + 1
};

static uint32_t env_u32(const char *name, uint32_t dflt)
{
    const char *v = getenv(name);
    if (!v || !*v) return dflt;
    return (uint32_t)strtoul(v, nullptr, 10);
}

// ---------------------------------------------------------------------------------------------------
extern "C" int gatb_version(void) { return GATB_VERSION; }

extern "C" int gatb_create(int device, gatb_ctx **out)
{
    if (!out) return fail(nullptr, GATB_ERR_INVALID, "gatb_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, GATB_ERR_CUDA,
                    std::string("gatb_create: no CUDA device (") + cudaGetErrorString(e) +
                        "); gat_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(nullptr, GATB_ERR_INVALID, "gatb_create: bad device index");
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail(nullptr, GATB_ERR_CUDA, cudaGetErrorString(e));
    gatb_ctx *ctx = new gatb_ctx();
    ctx->device = device;
    e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete ctx; return fail(nullptr, GATB_ERR_CUDA, cudaGetErrorString(e)); }
    ctx->stream = ctx->own_stream;
    e = cudaStreamCreateWithFlags(&ctx->upload_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->build_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2 && e == cudaSuccess; i++) {
        e = cudaEventCreateWithFlags(&ctx->ev_counted[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaMallocHost(&ctx->err_slots, 256 * 4 * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMallocHost(&ctx->small_stage, 256 * SMALL_STAGE_BYTES);
    if (e != cudaSuccess) { cudaStreamDestroy(ctx->own_stream); delete ctx; return fail(nullptr, GATB_ERR_CUDA, cudaGetErrorString(e)); }
    for (int i = 255; i >= 0; i--) ctx->err_free.push_back(i);
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    ctx->count_threads = (int)std::min(1024u, std::max(32u, env_u32("GATB_COUNT_THREADS", 1024) / 32 * 32));
    ctx->schunk_max = env_u32("GATB_SCHUNK", 0);
    ctx->kgrp_max = env_u32("GATB_KEY_GROUP", 0);
    ctx->trace = env_u32("GATB_TRACE", 0) != 0;
    ctx->stats_stream = env_u32("GATB_STATS_STREAM", 1) != 0;
    ctx->scratch = new BatchScratch();
    ctx->blocks = new BlockCache();
    ctx->batch = env_u32("GATB_BATCH", 0);
    *out = ctx;
    return GATB_OK;
}

extern "C" void gatb_destroy(gatb_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    delete ctx->scratch;
    if (ctx->blocks) { ctx->blocks->drop(ctx->upload_stream); cudaStreamSynchronize(ctx->upload_stream); delete ctx->blocks; }
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->upload_stream) cudaStreamDestroy(ctx->upload_stream);
    if (ctx->build_stream) cudaStreamDestroy(ctx->build_stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    for (int i = 0; i < 2; i++) {
        if (ctx->ev_counted[i]) cudaEventDestroy(ctx->ev_counted[i]);
        if (ctx->ev_copied[i]) cudaEventDestroy(ctx->ev_copied[i]);
    }
    if (ctx->err_slots) cudaFreeHost(ctx->err_slots);
    if (ctx->small_stage) cudaFreeHost(ctx->small_stage);
    delete ctx;
}

extern "C" const char *gatb_last_error(gatb_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

extern "C" int gatb_set_stream(gatb_ctx *ctx, void *cuda_stream)
{
    if (!ctx) return GATB_ERR_INVALID;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);           // buffers allocated on the old stream are complete
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return GATB_OK;
}

extern "C" int gatb_synchronize(gatb_ctx *ctx)
{
    if (!ctx) return GATB_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return GATB_OK;
}

extern "C" uint64_t gatb_launch_count(gatb_ctx *ctx) { return ctx ? ctx->launches : 0; }

extern "C" int gatb_profile(gatb_ctx *ctx, int enable)
{
    if (!ctx) return GATB_ERR_INVALID;
    ctx->profiling = enable != 0;
    return GATB_OK;
}

extern "C" int gatb_profile_read(gatb_ctx *ctx, double *ms, uint64_t *launches)
{
    if (!ctx || !ms || !launches) return GATB_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < PROF_NCLS; i++) { ms[i] = 0; launches[i] = 0; }
    for (auto &sp : ctx->spans) {
        float t = 0;
        cudaEventElapsedTime(&t, sp.a, sp.b);
        ms[sp.cls] += t; launches[sp.cls]++;
        cudaEventDestroy(sp.a); cudaEventDestroy(sp.b);
    }
    ctx->spans.clear();
    return GATB_OK;
}

extern "C" int gatb_set_batch_size(gatb_ctx *ctx, uint32_t batch)
{
    if (!ctx) return GATB_ERR_INVALID;
    ctx->batch = batch;
    return GATB_OK;
}

// ---------------------------------------------------------------------------------------------------
// validation helpers
static int check_lists(gatb_ctx *ctx, const char *what, uint64_t n_lists, const uint64_t *offs,
                       const uint32_t *start, const uint32_t *end)
{
    if (!offs) return fail(ctx, GATB_ERR_INVALID, std::string(what) + ": offsets are NULL");
    if (offs[0] != 0) return fail(ctx, GATB_ERR_INVALID, std::string(what) + ": offsets must start at 0");
    for (uint64_t l = 0; l < n_lists; l++) {
        if (offs[l + 1] < offs[l]) return fail(ctx, GATB_ERR_INVALID, std::string(what) + ": offsets not monotone");
        for (uint64_t i = offs[l]; i < offs[l + 1]; i++) {
            if (end[i] >= 0x80000000u) return fail(ctx, GATB_ERR_RANGE, std::string(what) + ": coordinate >= 2^31");
            if (start[i] >= end[i]) return fail(ctx, GATB_ERR_INVALID, std::string(what) + ": empty or inverted segment (list not normalized)");
            if (i > offs[l] && end[i - 1] > start[i])
                return fail(ctx, GATB_ERR_INVALID, std::string(what) + ": list not sorted/normalized");
        }
    }
    return GATB_OK;
}

// ---------------------------------------------------------------------------------------------------
// annotations
struct gatb_annotations {
    gatb_ctx *ctx = nullptr;
    uint32_t n_annot = 0, n_keys = 0, n_groups = 0, ka = 1;
    uint64_t n_intervals = 0;
    uint64_t n_boff = 0, capacity = 0;
    uint64_t n_entries = 0;             // entries the built index holds (padding included)
    bool has_long = false;              // it holds intervals of >= 2^20 - 1 bases
    std::vector<KeyBins> h_keybins;
    DevBuf<KeyBins> keybins;
    DevBuf<uint32_t> boff;
    DevBuf<uint4> brec;
    DevBuf<uint2> civ;
    DevBuf<uint2> cent;
    DevBuf<uint32_t> cprev;
    DevBuf<uint32_t> key_ws_nseg;
    bool has_nseg = false;
    // kept until the build has been checked (annotations_finish): the raw lists on the device, so that an
    // index that outgrew the estimated capacity can be rebuilt at its exact size without the caller's arrays
    DevBuf<uint64_t> d_offs;
    DevBuf<uint32_t> d_start, d_end, d_err, d_jmax;
    // where the build reads the lists: the copies above, or device lists owned by the caller (gatb_lists)
    const uint64_t *src_offs = nullptr;
    const uint32_t *src_start = nullptr, *src_end = nullptr;
    uint32_t jmax_all = 0;
    DevBuf<unsigned long long> d_total;
    DevBuf<uint8_t> scan_tmp;
    // asynchronous create: `ready` is recorded on the upload stream after the index build; until the
    // first wait the validation words (pinned, err_slot) have not been looked at
    cudaEvent_t ready = nullptr;
    int err_slot = -1;
    bool pending = false;
    int status = GATB_OK;
    ~gatb_annotations()
    {
        if (ready) { cudaEventSynchronize(ready); cudaEventDestroy(ready); }
        if (err_slot >= 0) ctx->err_free.push_back(err_slot);
    }
};

static void build_params(const gatb_annotations *a, BuildBinsParams &bp)
{
    memset(&bp, 0, sizeof(bp));
    bp.offs = a->src_offs; bp.start = a->src_start; bp.end = a->src_end; bp.n_intervals = a->n_intervals;
    bp.keybins = a->keybins.p; bp.key_jmax = a->d_jmax.p; bp.jmax_all = a->jmax_all; bp.boff = a->boff.p; bp.brec = a->brec.p; bp.n_boff = a->n_boff;
    bp.cent = a->cent.p; bp.civ = a->civ.p; bp.cprev = a->cprev.p; bp.capacity = a->capacity;
    bp.n_annot = a->n_annot; bp.n_keys = a->n_keys; bp.n_groups = a->n_groups; bp.ka = a->ka;
    bp.a_begin = 0; bp.a_count = a->n_annot;
    bp.error = a->d_err.p; bp.has_long = a->d_err.p + 1; bp.total = a->d_total.p;
}

// queue on `st`: scan + fill of the index (the per-bin counts are in place), the read-back of the validation
// word and of the number of entries the index needs, and the `ready` event
static cudaError_t annotations_build_finish(gatb_annotations *a, cudaStream_t st)
{
    gatb_ctx *ctx = a->ctx;
    uint32_t *slot = ctx->err_slots + 4 * a->err_slot;
    BuildBinsParams bp;
    build_params(a, bp);
    cudaError_t e;
    {
        ProfScope ps(ctx, PROF_OTHER, st);
        ctx->launches += 6;                 // even, scan (2), total, fill, pad, records
        e = launch_bins_finish(st, bp, a->scan_tmp.p, a->scan_tmp.n);
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(slot, a->d_err.p, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(slot + 2, a->d_total.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaEventRecord(a->ready, st);
    return e;
}

// queue (on the upload stream) the whole construction of the grid index from the device copies of the lists
static cudaError_t annotations_build(gatb_annotations *a)
{
    gatb_ctx *ctx = a->ctx;
    cudaStream_t st = ctx->upload_stream;
    cudaError_t e = cudaMemsetAsync(a->d_err.p, 0, 2 * sizeof(uint32_t), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(a->d_total.p, 0, sizeof(unsigned long long), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(a->boff.p, 0, 2 * (a->n_boff + 1) * sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    BuildBinsParams bp;
    build_params(a, bp);
    { ProfScope ps(ctx, PROF_OTHER, st); e = launch_bins_count(st, bp); }
    if (e == cudaSuccess) e = annotations_build_finish(a, st);
    return e;
}

// host-blocking: the asynchronous build has finished; -> validation result.  An index that needed more
// entries than estimated is rebuilt here at its exact size.
static int annotations_finish(gatb_annotations *a)
{
    if (!a->pending) return a->status;
    gatb_ctx *ctx = a->ctx;
    a->pending = false;
    const uint32_t *slot = ctx->err_slots + 4 * a->err_slot;
    cudaStream_t saved = tl_stream;
    tl_stream = ctx->upload_stream;
    cudaError_t e = cudaEventSynchronize(a->ready);
    uint32_t h_err = slot[0];
    memcpy(&a->n_entries, slot + 2, sizeof(uint64_t));
    a->has_long = slot[1] != 0;
    if (e == cudaSuccess && !(h_err & 3u) && (h_err & 4u)) {
        unsigned long long need;
        memcpy(&need, slot + 2, sizeof(need));
        if (need > 0xfffffff0ull) {
            tl_stream = saved;
            return a->status = fail(ctx, GATB_ERR_INVALID, "annotations: index needs 2^32 or more entries");
        }
        a->capacity = need;                 // (even: every bin has an even number of slots)
        e = a->civ.alloc(need + 2);
        if (e == cudaSuccess) e = a->cent.alloc(need + 2);
        if (e == cudaSuccess) e = a->cprev.alloc(need + 2);
        if (e == cudaSuccess) e = annotations_build(a);
        if (e == cudaSuccess) e = cudaEventSynchronize(a->ready);
        h_err = slot[0];
        memcpy(&a->n_entries, slot + 2, sizeof(uint64_t));
        a->has_long = slot[1] != 0;
    }
    // the raw lists and the scan scratch are no longer needed (freed in upload-stream order)
    a->d_offs.release(); a->d_start.release(); a->d_end.release(); a->d_err.release(); a->d_total.release();
    a->d_jmax.release();
    a->scan_tmp.release();
    tl_stream = saved;
    if (e != cudaSuccess) return a->status = fail(ctx, GATB_ERR_CUDA, cudaGetErrorString(e));
    if (h_err & 1u) return a->status = fail(ctx, GATB_ERR_RANGE, "annotations: coordinate >= 2^31");
    if (h_err & 2u) return a->status = fail(ctx, GATB_ERR_INVALID, "annotations: empty or inverted segment, or list not sorted/normalized");
    if (h_err) return a->status = fail(ctx, GATB_ERR_CUDA, "annotations: index build failed");
    return a->status = GATB_OK;
}

static inline uint32_t floor_log2(uint64_t x) { uint32_t l = 0; while (x >>= 1) l++; return l; }

// The lists of an annotation set come either from the host (start / end: copied up in chunks while the build
// counts behind them) or from device lists the caller owns (dev_*: read in place; `last_end[l]` = end of list l's
// last interval and `mean_len` then stand in for the host arrays; the caller keeps the lists alive until the
// build has been waited for).
static int annotations_create_common(gatb_ctx *ctx, int n_annot, int n_keys, const uint64_t *offs,
                                     const uint32_t *start, const uint32_t *end, const uint32_t *last_end, uint64_t mean_len_dev,
                                     const uint64_t *dev_offs, const uint32_t *dev_start, const uint32_t *dev_end,
                                     const uint32_t *key_ws_nseg, gatb_annotations **out)
{
    if (!ctx || !out) return GATB_ERR_INVALID;
    *out = nullptr;
    if (n_annot <= 0 || n_keys <= 0) return fail(ctx, GATB_ERR_INVALID, "annotations: need >=1 track and >=1 key");
    const uint64_t n_lists = (uint64_t)n_annot * n_keys;
    const bool from_device = dev_offs != nullptr;
    // offsets are checked here; the intervals themselves (range, order, normalisation) on the GPU
    if (!offs || (!from_device && (!start || !end))) return fail(ctx, GATB_ERR_INVALID, "annotations: NULL array");
    if (offs[0] != 0) return fail(ctx, GATB_ERR_INVALID, "annotations: offsets must start at 0");
    for (uint64_t l = 0; l < n_lists; l++)
        if (offs[l + 1] < offs[l]) return fail(ctx, GATB_ERR_INVALID, "annotations: offsets not monotone");
    const uint64_t n_iv = offs[n_lists];
    if (n_iv > 0xffffffffull) return fail(ctx, GATB_ERR_INVALID, "annotations: more than 2^32 intervals");
    CU(ctx, cudaSetDevice(ctx->device));
    if (ctx->err_free.empty()) return fail(ctx, GATB_ERR_INVALID, "annotations: more than 256 sets pending validation");
    tl_stream = ctx->upload_stream;       // every allocation, copy and free below is ordered on the upload stream

    const auto t_begin = std::chrono::steady_clock::now();
    auto since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
    double t_plan = 0, t_alloc = 0, t_queue = 0;
    const uint32_t A = (uint32_t)n_annot, K = (uint32_t)n_keys;
    const uint32_t ka = std::min(A, std::min(GROUP_TRACKS_MAX, std::max(1u, env_u32("GATB_GROUP_TRACKS", GROUP_TRACKS_MAX))));
    const uint32_t G = (A + ka - 1) / ka;

    // Bin width: about the mean interval length (estimated from a few thousand intervals; any value is
    // correct, it only trades entries per interval against entries per bin), but per key no more than
    // ~4 bins per interval, so that sparse lists do not pay for empty bins.
    uint32_t shift = env_u32("GATB_BIN_SHIFT", 0);
    uint64_t mean_len = std::max<uint64_t>(1, mean_len_dev);
    if (n_iv && !from_device) {
        const uint64_t step = std::max<uint64_t>(1, n_iv / 4096);
        uint64_t sum = 0, cnt = 0;
        for (uint64_t i = 0; i < n_iv; i += step) { sum += (end[i] > start[i]) ? end[i] - start[i] : 0u; cnt++; }
        mean_len = std::max<uint64_t>(1, sum / cnt);
    }
    // about half the mean interval length: a segment tests its true overlaps (the C list of its first bin holds
    // little else) plus the intervals starting within ~W/2 of either end, while an interval is stored
    // 1 + length / W times (measured on the benchmark shape, mean length 1.4 kb: W = 256 / 512 / 1024 / 2048 ->
    // 14.5 / 15.8 / 18.9 / 25.4 entries tested per segment for 11.2 true overlaps, index 1.2 / 0.68 / 0.42 /
    // 0.29 GB, counting kernel 1.40 / 1.40 / 1.47 / 1.70 ms; profiles/r02_bin_width_sweep.txt)
    if (shift == 0) shift = floor_log2(mean_len) > 4 ? floor_log2(mean_len) - 1 : 4;
    shift = std::min(20u, std::max(4u, shift));
    gatb_annotations *a = new gatb_annotations();
    a->ctx = ctx; a->n_annot = A; a->n_keys = K; a->n_groups = G; a->ka = ka;
    a->n_intervals = n_iv;
    a->h_keybins.resize((size_t)G * K);
    uint64_t n_boff = 0;
    double est = 0;
    std::vector<uint32_t> jmax(K, 0);
    for (uint32_t t = 0; t < A; t++)
        for (uint32_t k = 0; k < K; k++)
            jmax[k] = std::max(jmax[k], (uint32_t)(offs[(uint64_t)t * K + k + 1] - offs[(uint64_t)t * K + k]));
    for (uint32_t k = 0; k < K; k++) a->jmax_all = std::max(a->jmax_all, jmax[k]);
    for (uint32_t g = 0; g < G; g++)
        for (uint32_t k = 0; k < K; k++) {
            uint64_t n = 0;
            uint32_t extent = 0;
            for (uint32_t t = g * ka; t < std::min(A, (g + 1) * ka); t++) {
                const uint64_t l = (uint64_t)t * K + k;
                if (offs[l + 1] > offs[l]) { n += offs[l + 1] - offs[l]; extent = std::max(extent, from_device ? last_end[l] : end[offs[l + 1] - 1]); }
            }
            KeyBins &kb = a->h_keybins[(size_t)g * K + k];
            kb.base = n_boff; kb.nbins = 0; kb.shift = shift;
            if (n == 0 || extent == 0) continue;
            extent = std::min(extent, 0x7fffffffu);            // (larger coordinates fail validation)
            uint32_t sh = shift;
            while (sh < 20 && ((uint64_t)(extent - 1) >> sh) + 1 > 4 * n + 16) sh++;
            kb.shift = sh;
            kb.nbins = (uint32_t)(((uint64_t)(extent - 1) >> sh) + 1);
            n_boff += (uint64_t)kb.nbins + 1;
            est += (double)n * (1.0 + (double)mean_len / (double)(1ull << sh));
        }
    if (n_boff > 0x3ffffff0ull) { delete a; return fail(ctx, GATB_ERR_INVALID, "annotations: index too large"); }
    a->n_boff = n_boff;
    // (+ up to one padding slot per list, two lists per bin: lists hold an even number of entries)
    a->capacity = (uint64_t)(est * 1.25) + n_boff + 4096;
    if (env_u32("GATB_INDEX_CAPACITY", 0)) a->capacity = env_u32("GATB_INDEX_CAPACITY", 0);    // (tests: forces the rebuild)
    a->capacity = (a->capacity + 1) & ~(uint64_t)1;

    t_plan = since();
    cudaStream_t st = ctx->upload_stream;
    a->err_slot = ctx->err_free.back();
    ctx->err_free.pop_back();
    memset(ctx->err_slots + 4 * a->err_slot, 0, 4 * sizeof(uint32_t));
    // the small host-built tables first (pageable memory: staged before the call returns), then the
    // caller's arrays, which must stay valid until gatb_annotations_wait() or the first use returns
    // (staged through the set's pinned slot when they fit: truly asynchronous copies)
    const size_t kb_bytes = a->h_keybins.size() * sizeof(KeyBins), k_bytes = (size_t)K * sizeof(uint32_t);
    const void *src_kb = a->h_keybins.data(), *src_nseg = key_ws_nseg, *src_jmax = jmax.data();
    if (kb_bytes + 2 * k_bytes <= SMALL_STAGE_BYTES) {
        uint8_t *stage = ctx->small_stage + (size_t)a->err_slot * SMALL_STAGE_BYTES;
        memcpy(stage, src_kb, kb_bytes); src_kb = stage;
        memcpy(stage + kb_bytes, src_jmax, k_bytes); src_jmax = stage + kb_bytes;
        if (key_ws_nseg) { memcpy(stage + kb_bytes + k_bytes, key_ws_nseg, k_bytes); src_nseg = stage + kb_bytes + k_bytes; }
    }
    cudaError_t e = a->keybins.upload((const KeyBins *)src_kb, a->h_keybins.size(), st);
    if (e == cudaSuccess && key_ws_nseg) { e = a->key_ws_nseg.upload((const uint32_t *)src_nseg, K, st); a->has_nseg = true; }
    if (e == cudaSuccess) e = a->d_jmax.upload((const uint32_t *)src_jmax, K, st);
    const double t_small = since();
    uint64_t pool_reserved0 = 0, pool_used0 = 0, pool_reserved1 = 0, pool_used1 = 0;
    cudaMemPool_t pool = nullptr;
    if (ctx->trace && cudaDeviceGetDefaultMemPool(&pool, ctx->device) == cudaSuccess) {
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &pool_reserved0);
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &pool_used0);
    }
    if (e == cudaSuccess) e = a->boff.alloc_cached(ctx->blocks, 2 * (n_boff + 1));
    if (e == cudaSuccess) e = a->brec.alloc_cached(ctx->blocks, std::max<uint64_t>(n_boff, 1));
    if (e == cudaSuccess) e = a->civ.alloc_cached(ctx->blocks, a->capacity + 2);
    if (e == cudaSuccess) e = a->cent.alloc_cached(ctx->blocks, a->capacity + 2);
    if (e == cudaSuccess) e = a->cprev.alloc_cached(ctx->blocks, a->capacity + 2);
    if (e == cudaSuccess) e = a->scan_tmp.alloc(build_bins_scan_bytes(n_boff));
    const double t_index_alloc = since();
    if (ctx->trace && pool) {
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &pool_reserved1);
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &pool_used1);
    }
    if (from_device) { a->src_offs = dev_offs; a->src_start = dev_start; a->src_end = dev_end; }
    else {
        if (e == cudaSuccess) e = a->d_offs.upload(offs, n_lists + 1, st);
        if (e == cudaSuccess) e = a->d_start.alloc_cached(ctx->blocks, n_iv);
        if (e == cudaSuccess) e = a->d_end.alloc_cached(ctx->blocks, n_iv);
        a->src_offs = a->d_offs.p; a->src_start = a->d_start.p; a->src_end = a->d_end.p;
    }
    if (e == cudaSuccess) e = a->d_err.alloc(2);
    if (e == cudaSuccess) e = a->d_total.alloc(1);
    const double t_raw_alloc = since();
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&a->ready, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMemsetAsync(a->d_err.p, 0, 2 * sizeof(uint32_t), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(a->d_total.p, 0, sizeof(unsigned long long), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(a->boff.p, 0, 2 * (n_boff + 1) * sizeof(uint32_t), st);
    t_alloc = since();
    // The intervals go up in chunks of tracks; the build stream counts the bin entries of a chunk (step 1 of
    // the build) while the next chunk is still on the bus, and runs scan + fill behind the last one.
    {
        const uint32_t n_chunks = (n_iv >= (4u << 20) && !from_device) ? std::min(4u, A) : 1u;
        BuildBinsParams bp;
        build_params(a, bp);
        for (uint32_t c = 0; c < n_chunks && e == cudaSuccess; c++) {
            const uint32_t a0 = (uint32_t)((uint64_t)A * c / n_chunks), a1 = (uint32_t)((uint64_t)A * (c + 1) / n_chunks);
            const uint64_t i0 = offs[(uint64_t)a0 * K], i1 = offs[(uint64_t)a1 * K];
            if (i1 > i0 && !from_device) {
                e = cudaMemcpyAsync(a->d_start.p + i0, start + i0, (i1 - i0) * sizeof(uint32_t), cudaMemcpyHostToDevice, st);
                if (e == cudaSuccess) e = cudaMemcpyAsync(a->d_end.p + i0, end + i0, (i1 - i0) * sizeof(uint32_t), cudaMemcpyHostToDevice, st);
            }
            cudaEvent_t ev = nullptr;
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventRecord(ev, st);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->build_stream, ev, 0);
            if (ev) cudaEventDestroy(ev);           // (released once it has completed)
            bp.a_begin = a0; bp.a_count = a1 - a0;
            if (e == cudaSuccess) { ProfScope ps(ctx, PROF_OTHER, ctx->build_stream); e = launch_bins_count(ctx->build_stream, bp); }
        }
        if (e == cudaSuccess) e = annotations_build_finish(a, ctx->build_stream);
    }
    if (e != cudaSuccess) {
        cudaStreamSynchronize(st); cudaStreamSynchronize(ctx->build_stream);
        delete a;
        return fail(ctx, GATB_ERR_CUDA, cudaGetErrorString(e));
    }
    t_queue = since();
    if (ctx->trace)
        fprintf(stderr, "gatb_annotations_create: geometry %.2f ms, small uploads %.2f, index allocations %.2f, raw list allocations "
                        "%.2f, event + memsets %.2f, copies + build queued %.2f\n",
                t_plan, t_small, t_index_alloc, t_raw_alloc, t_alloc, t_queue);
    if (ctx->trace)
        fprintf(stderr, "gatb_annotations_create: pool before the index allocations: reserved %.0f MB, used %.0f MB; after: reserved %.0f MB, used %.0f MB\n",
                pool_reserved0 / 1e6, pool_used0 / 1e6, pool_reserved1 / 1e6, pool_used1 / 1e6);
    a->pending = true;
    *out = a;
    return GATB_OK;
}

extern "C" int gatb_annotations_create_async(gatb_ctx *ctx, int n_annot, int n_keys, const uint64_t *offs,
                                             const uint32_t *start, const uint32_t *end, const uint32_t *key_ws_nseg,
                                             gatb_annotations **out)
{
    return annotations_create_common(ctx, n_annot, n_keys, offs, start, end, nullptr, 0, nullptr, nullptr, nullptr, key_ws_nseg, out);
}

extern "C" int gatb_annotations_wait(gatb_annotations *a)
{
    if (!a) return GATB_ERR_INVALID;
    cudaSetDevice(a->ctx->device);
    return annotations_finish(a);
}

extern "C" int gatb_annotations_create(gatb_ctx *ctx, int n_annot, int n_keys, const uint64_t *offs,
                                       const uint32_t *start, const uint32_t *end, const uint32_t *key_ws_nseg,
                                       gatb_annotations **out)
{
    int rc = gatb_annotations_create_async(ctx, n_annot, n_keys, offs, start, end, key_ws_nseg, out);
    if (rc) return rc;
    rc = annotations_finish(*out);
    if (rc) {
        tl_stream = ctx->stream;
        delete *out;
        *out = nullptr;
    }
    return rc;
}

extern "C" void gatb_annotations_destroy(gatb_annotations *a)
{
    if (!a) return;
    gatb_ctx *ctx = a->ctx;
    cudaSetDevice(ctx->device);
    if (a->pending) annotations_finish(a);
    // The index was allocated on the upload stream and last read on the compute stream: free it on the
    // upload stream once the compute stream has got this far, so that the next set's allocations (same
    // stream) re-use the memory without the pool having to reconcile two streams.
    cudaEvent_t ev = nullptr;
    if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) == cudaSuccess) {
        cudaEventRecord(ev, ctx->stream);
        cudaStreamWaitEvent(ctx->upload_stream, ev, 0);
        cudaEventDestroy(ev);
    } else cudaStreamSynchronize(ctx->stream);
    delete a;
}

// fill the annotation side of CountParams and pick the sample chunk
static int count_params_annos(const gatb_annotations *a, uint32_t n_samples, bool density, CountParams &p)
{
    gatb_ctx *ctx = a->ctx;
    p.keybins = a->keybins.p; p.boff = a->boff.p; p.coff_base = a->n_boff + 1; p.brec = a->brec.p; p.cent = a->cent.p; p.civ = a->civ.p; p.cprev = a->cprev.p; p.sentinel = (uint32_t)a->capacity; p.has_long = a->has_long ? 1u : 0u;
    p.key_ws_nseg = a->has_nseg ? a->key_ws_nseg.p : nullptr;
    p.n_annot = a->n_annot; p.n_keys = a->n_keys; p.n_groups = a->n_groups; p.ka = a->ka;
    p.n_samples = n_samples;
    // samples per CTA: what shared memory allows next to the staging and ITEM_TABLE_BYTES of item tables,
    // then as few whole waves of CTAs as that needs
    const size_t ITEM_TABLE_BYTES = 24576;
    const size_t cell = density ? 20u : 4u;
    const size_t fixed = count_smem_bytes(0, 0, 0, ctx->count_threads, density) + ITEM_TABLE_BYTES + 1024;
    const size_t room = ctx->smem_optin > fixed ? ctx->smem_optin - fixed : 0;
    uint32_t smax = (uint32_t)std::min<size_t>(room / (cell * a->ka), 2048);
    if (ctx->schunk_max) smax = std::min(smax, ctx->schunk_max);
    if (smax == 0) return fail(ctx, GATB_ERR_INVALID, "count: accumulators of one sample do not fit shared memory");
    const uint64_t per_wave = std::max<uint64_t>(1, (uint64_t)ctx->sm_count / a->n_groups);
    uint64_t chunks = (n_samples + smax - 1) / smax;
    if (n_samples >= per_wave) chunks = (chunks + per_wave - 1) / per_wave * per_wave;
    p.schunk = (uint32_t)std::max<uint64_t>(1, (n_samples + chunks - 1) / chunks);
    p.kgrp = (uint32_t)std::max<size_t>(1, std::min<size_t>(a->n_keys, ITEM_TABLE_BYTES / (8u * p.schunk + 8u)));
    if (ctx->kgrp_max) p.kgrp = std::min(p.kgrp, ctx->kgrp_max);
    return GATB_OK;
}

// ---------------------------------------------------------------------------------------------------
// counting of explicit lists (observed counts, same-placement parity)
extern "C" int gatb_count_lists(gatb_ctx *ctx, const gatb_annotations *annos, int n_counters, const int32_t *counters,
                                uint64_t n_samples, const uint64_t *offs, const uint32_t *start, const uint32_t *end,
                                const uint8_t *key_present, double *out)
{
    if (!ctx || !annos || !counters || !out || n_counters <= 0) return GATB_ERR_INVALID;
    if (n_samples == 0) return GATB_OK;
    if (n_samples > 0x7fffffffull) return fail(ctx, GATB_ERR_INVALID, "count_lists: too many samples");
    const uint32_t K = annos->n_keys, A = annos->n_annot;
    int rc = check_lists(ctx, "segments", n_samples * K, offs, start, end);
    if (rc) return rc;
    for (int c = 0; c < n_counters; c++) {
        if (counters[c] < 0 || counters[c] >= GATB_NCOUNTERS) return fail(ctx, GATB_ERR_INVALID, "unknown counter id");
        if (counters[c] == GATB_NUCLEOTIDE_DENSITY && !annos->has_nseg)
            return fail(ctx, GATB_ERR_INVALID, "nucleotide-density needs key_ws_nseg at gatb_annotations_create");
    }
    CU(ctx, cudaSetDevice(ctx->device));
    rc = annotations_finish(const_cast<gatb_annotations *>(annos));
    if (rc) return rc;
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;

    // capacity layout: key k of sample s at s*stride + key_base[k]
    std::vector<uint64_t> key_base(K);
    std::vector<uint32_t> cap(K, 0);
    for (uint64_t s = 0; s < n_samples; s++)
        for (uint32_t k = 0; k < K; k++)
            cap[k] = std::max<uint32_t>(cap[k], (uint32_t)(offs[s * K + k + 1] - offs[s * K + k]));
    uint64_t stride = 0;
    for (uint32_t k = 0; k < K; k++) {
        if (cap[k] >= (1u << 24)) return fail(ctx, GATB_ERR_INVALID, "count_lists: 2^24 or more segments on one key");
        key_base[k] = stride; stride += cap[k];
    }
    if (stride == 0) stride = 1;
    std::vector<uint64_t> packed(n_samples * stride, 0);
    std::vector<uint32_t> counts(n_samples * K);
    for (uint64_t s = 0; s < n_samples; s++)
        for (uint32_t k = 0; k < K; k++) {
            const uint64_t b = offs[s * K + k], n = offs[s * K + k + 1] - b;
            counts[s * K + k] = (uint32_t)n;
            uint64_t *dst = packed.data() + s * stride + key_base[k];
            for (uint64_t i = 0; i < n; i++) dst[i] = pack_seg(start[b + i], end[b + i]);
        }
    DevBuf<uint64_t> d_packed, d_base;
    DevBuf<uint32_t> d_n, d_out;
    DevBuf<uint8_t> d_present;
    DevBuf<double> d_outf;
    CU(ctx, d_packed.upload(packed.data(), packed.size(), st));
    CU(ctx, d_base.upload(key_base.data(), K, st));
    CU(ctx, d_n.upload(counts.data(), counts.size(), st));
    if (key_present) CU(ctx, d_present.upload(key_present, n_samples * K, st));
    CU(ctx, d_out.alloc(n_samples * A));
    CU(ctx, d_outf.alloc(n_samples * A));

    CountParams p;
    memset(&p, 0, sizeof(p));
    p.placed = d_packed.p; p.sample_stride = stride; p.key_base = d_base.p; p.placed_n = d_n.p;
    p.key_present = key_present ? d_present.p : nullptr;
    p.out_u32 = d_out.p; p.out_f64 = d_outf.p;

    std::vector<uint32_t> h_u(n_samples * A);
    for (int c = 0; c < n_counters; c++) {
        rc = count_params_annos(annos, (uint32_t)n_samples, counters[c] == GATB_NUCLEOTIDE_DENSITY, p);
        if (rc) return rc;
        { ProfScope ps(ctx, PROF_COUNT); CU(ctx, launch_count(st, counters[c], p, ctx->count_threads)); }
        double *o = out + (uint64_t)c * n_samples * A;
        if (counters[c] == GATB_NUCLEOTIDE_DENSITY) {
            CU(ctx, cudaMemcpyAsync(o, d_outf.p, n_samples * A * sizeof(double), cudaMemcpyDeviceToHost, st));
            CU(ctx, cudaStreamSynchronize(st));
        } else {
            CU(ctx, cudaMemcpyAsync(h_u.data(), d_out.p, n_samples * A * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
            CU(ctx, cudaStreamSynchronize(st));
            for (uint64_t i = 0; i < n_samples * A; i++) o[i] = (double)h_u[i];
        }
    }
    return GATB_OK;
}

// ---------------------------------------------------------------------------------------------------
// sampler
struct gatb_sampler {
    gatb_ctx *ctx = nullptr;
    uint32_t n_units = 0, n_contigs = 0;
    bool has_iso = false;
    bool one_piece = false;             // every unit's workspace is one piece (place_kernel<true>)
    int kind = 0;                       // 0 SamplerAnnotator, 1 SamplerSegments, 2 SamplerShift
    double shift_radius = 2.0;          // SamplerShift(radius, extension), gat/Engine.pyx:1021-1026
    int32_t shift_extension = 0;
    std::vector<UnitDesc> h_units;
    std::vector<uint64_t> h_contig_base;
    std::vector<uint32_t> h_contig_cap;
    uint64_t unit_stride = 0, placed_stride = 0;
    DevBuf<UnitDesc> units;
    DevBuf<uint32_t> order;
    DevBuf<uint32_t> ws_start, ws_end, ws_cuminc, len_tab;
    DevBuf<uint32_t> seg_start, seg_end;  // the units' raw segments (preparation; SamplerShift moves them)
    DevBuf<uint32_t> contig_unit_off, contig_units;
    DevBuf<uint64_t> contig_base;
    DevBuf<unsigned long long> tally;     // [3]: placed segments, round-cap units, overflow units
    DevBuf<uint32_t> unit_over;           // [n_units]: unit overflowed its buffer in the current call
    DevBuf<uint32_t> ws_tab;              // bucket tables over the workspace pieces of units with many pieces
    bool no_hist = false;                 // created with nbuckets = 0: no length histogram (SamplerShift only)
};

// Buffer layout from the units' capacities (UnitDesc.cap): offsets of the unit buffers inside one sample's
// region, contig-level capacities, the heaviest-first unit order; uploads the descriptors.  *why is set
// (and nothing uploaded) when a contig would need too large a buffer.
#define TRY(x) do { if (e == cudaSuccess) e = (x); } while (0)
static cudaError_t sampler_layout(gatb_sampler *s, cudaStream_t st, const char **why)
{
    const uint32_t U = s->n_units, C = s->n_contigs;
    // buffer layout
    s->h_contig_base.assign(C, 0);
    s->h_contig_cap.assign(C, 0);
    std::vector<uint32_t> cu_off(C + 1, 0), cu(U);
    for (uint32_t u = 0; u < U; u++) cu_off[s->h_units[u].contig + 1]++;
    for (uint32_t c = 0; c < C; c++) cu_off[c + 1] += cu_off[c];
    {
        std::vector<uint32_t> fill(cu_off.begin(), cu_off.end() - 1);
        for (uint32_t u = 0; u < U; u++) cu[fill[s->h_units[u].contig]++] = u;
    }
    if (s->has_iso) {
        uint64_t o = 0;
        for (uint32_t u = 0; u < U; u++) { s->h_units[u].buf_off = o; o += s->h_units[u].cap; }
        s->unit_stride = o;
        uint64_t b = 0;
        for (uint32_t c = 0; c < C; c++) {
            uint64_t sum = 0;
            for (uint32_t k = cu_off[c]; k < cu_off[c + 1]; k++) sum += s->h_units[cu[k]].cap;
            s->h_contig_cap[c] = next_pow2((uint32_t)std::max<uint64_t>(sum, 1));
            s->h_contig_base[c] = b;
            b += s->h_contig_cap[c];
        }
        s->placed_stride = b;
    } else {
        uint64_t b = 0;
        for (uint32_t c = 0; c < C; c++) {
            uint32_t capc = 64;
            for (uint32_t k = cu_off[c]; k < cu_off[c + 1]; k++) capc = s->h_units[cu[k]].cap;
            s->h_contig_cap[c] = capc;
            s->h_contig_base[c] = b;
            for (uint32_t k = cu_off[c]; k < cu_off[c + 1]; k++) s->h_units[cu[k]].buf_off = b;
            b += capc;
        }
        s->placed_stride = b;
        s->unit_stride = 0;
    }
    for (uint32_t c = 0; c < C; c++)
        if (s->h_contig_cap[c] > (1u << 24)) { *why = "sampler: more than 2^23 segments on one contig"; return cudaSuccess; }
    std::vector<uint32_t> order(U);
    for (uint32_t u = 0; u < U; u++) order[u] = u;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return s->h_units[a].tab_n > s->h_units[b].tab_n; });
    cudaError_t e = cudaSuccess;
    TRY(cudaMemcpyAsync(s->units.p, s->h_units.data(), U * sizeof(UnitDesc), cudaMemcpyHostToDevice, st));
    TRY(s->order.upload(order.data(), U, st));
    TRY(s->contig_unit_off.upload(cu_off.data(), C + 1, st));
    TRY(s->contig_units.upload(cu.data(), U, st));
    TRY(s->contig_base.upload(s->h_contig_base.data(), C, st));
    TRY(cudaStreamSynchronize(st));         // (the host vectors above are the copies' sources)
    return e;
}
#undef TRY

extern "C" int gatb_sampler_create(gatb_ctx *ctx, int n_units, const int32_t *unit_contig, int n_contigs,
                                   int has_isochores,
                                   const uint64_t *seg_offs, const uint32_t *seg_start, const uint32_t *seg_end,
                                   const uint64_t *ws_offs, const uint32_t *ws_start, const uint32_t *ws_end,
                                   uint32_t bucket_size, uint32_t nbuckets, gatb_sampler **out)
{
    if (!ctx || !out) return GATB_ERR_INVALID;
    *out = nullptr;
    if (n_units <= 0 || n_contigs <= 0 || !unit_contig) return fail(ctx, GATB_ERR_INVALID, "sampler: need >=1 unit");
    const uint32_t U = (uint32_t)n_units, C = (uint32_t)n_contigs;
    const auto t_begin = std::chrono::steady_clock::now();
    auto since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
    int rc = check_lists(ctx, "segments", U, seg_offs, seg_start, seg_end);
    if (rc) return rc;
    rc = check_lists(ctx, "workspace", U, ws_offs, ws_start, ws_end);
    if (rc) return rc;
    if (seg_offs[U] > 0x7fffffffull || ws_offs[U] > 0x7fffffffull)
        return fail(ctx, GATB_ERR_INVALID, "sampler: more than 2^31 segments");
    std::vector<uint32_t> per_contig(C, 0);
    for (uint32_t u = 0; u < U; u++) {
        if (unit_contig[u] < 0 || (uint32_t)unit_contig[u] >= C) return fail(ctx, GATB_ERR_INVALID, "sampler: unit_contig out of range");
        if (seg_offs[u + 1] == seg_offs[u] || ws_offs[u + 1] == ws_offs[u])
            return fail(ctx, GATB_ERR_INVALID, "sampler: units with empty segments or workspace must be skipped by the caller");
        per_contig[unit_contig[u]]++;
    }
    if (!has_isochores)
        for (uint32_t c = 0; c < C; c++)
            if (per_contig[c] > 1) return fail(ctx, GATB_ERR_INVALID, "sampler: several units per contig need has_isochores");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;

    gatb_sampler *s = new gatb_sampler();
    s->ctx = ctx; s->n_units = U; s->n_contigs = C; s->has_iso = has_isochores != 0;
    s->no_hist = nbuckets == 0;
    // workspace CDF (SegmentListSampler.__init__, gat/Engine.pyx:261-277) and unit descriptors
    std::vector<uint32_t> cuminc(ws_offs[U]);
    s->h_units.resize(U);
    std::vector<uint64_t> scratch_off(U);
    uint64_t scratch_total = 0, ws_tab_total = 0;
    for (uint32_t u = 0; u < U; u++) {
        UnitDesc &d = s->h_units[u];
        memset(&d, 0, sizeof(d));
        d.ws_off = (uint32_t)ws_offs[u]; d.ws_n = (uint32_t)(ws_offs[u + 1] - ws_offs[u]);
        uint64_t t = 0;
        for (uint64_t i = ws_offs[u]; i < ws_offs[u + 1]; i++) { t += ws_end[i] - ws_start[i]; cuminc[i] = (uint32_t)t; }
        if (t > 0xffffffffull) { delete s; return fail(ctx, GATB_ERR_RANGE, "sampler: workspace unit larger than 2^32 bases"); }
        d.ws_total = (uint32_t)t;
        d.seg_off = (uint32_t)seg_offs[u]; d.seg_n = (uint32_t)(seg_offs[u + 1] - seg_offs[u]);
        d.tab_off = d.seg_off;
        d.contig = (uint32_t)unit_contig[u];
        scratch_off[u] = scratch_total;
        scratch_total += next_pow2(std::max(d.seg_n, 1u));
        // bucket tables (common.cuh WS_NB): worth it from a handful of pieces on; the entries are 16-bit
        d.ws_tab_off = 0xffffffffu;
        if (d.ws_n >= 8 && d.ws_n < 65535 && d.ws_total >= 65536 && ws_end[ws_offs[u + 1] - 1] - ws_start[ws_offs[u]] >= 65536) {
            d.ws_tab_off = (uint32_t)ws_tab_total;
            ws_tab_total += 2 + (WS_NB + 1);        // words: two multipliers + 2 * (WS_NB + 1) 16-bit entries
        }
    }
    s->one_piece = std::all_of(s->h_units.begin(), s->h_units.end(), [](const UnitDesc &d) { return d.ws_n == 1; });
    const double t_host = since();
    DevBuf<uint32_t> &d_seg_start = s->seg_start, &d_seg_end = s->seg_end;
    DevBuf<uint64_t> d_scratch, d_scratch_off;
    cudaError_t e = cudaSuccess;
#define TRY(x) do { if (e == cudaSuccess) e = (x); } while (0)
    TRY(d_seg_start.upload(seg_start, seg_offs[U], st));
    TRY(d_seg_end.upload(seg_end, seg_offs[U], st));
    TRY(s->ws_start.upload(ws_start, ws_offs[U], st));
    TRY(s->ws_end.upload(ws_end, ws_offs[U], st));
    TRY(s->ws_cuminc.upload(cuminc.data(), cuminc.size(), st));
    TRY(s->units.upload(s->h_units.data(), U, st));
    TRY(s->len_tab.alloc(seg_offs[U]));
    TRY(d_scratch.alloc(scratch_total));
    TRY(d_scratch_off.upload(scratch_off.data(), U, st));
    TRY(s->ws_tab.alloc(std::max<uint64_t>(ws_tab_total, 2)));
    const double t_uploads = since();
    if (e == cudaSuccess) {
        ProfScope ps(ctx, PROF_OTHER);
        launch_prep_units(st, s->units.p, U, d_seg_start.p, d_seg_end.p, s->ws_start.p, s->ws_end.p, s->ws_cuminc.p,
                          s->len_tab.p, d_scratch.p, d_scratch_off.p, bucket_size, nbuckets, s->ws_tab.p);
        e = cudaGetLastError();
    }
    TRY(cudaMemcpyAsync(s->h_units.data(), s->units.p, U * sizeof(UnitDesc), cudaMemcpyDeviceToHost, st));
    TRY(cudaStreamSynchronize(st));
    const double t_prep = since();
    if (e != cudaSuccess) { delete s; return fail(ctx, GATB_ERR_CUDA, cudaGetErrorString(e)); }
    for (uint32_t u = 0; u < U; u++)
        if (s->h_units[u].error) {
            delete s;
            return fail(ctx, GATB_ERR_TOO_LARGE,
                        "segment too large: increase nbuckets or bucket_size such that nbuckets * bucket_size > largest segment");
        }
    // (tests: GATB_PLACE_CAP_MAX clamps the estimated capacities so that the grow-and-repeat path runs)
    if (const uint32_t cap_max = env_u32("GATB_PLACE_CAP_MAX", 0))
        for (uint32_t u = 0; u < U; u++) s->h_units[u].cap = std::min(s->h_units[u].cap, next_pow2(std::max(cap_max, 64u)));
    uint64_t lsum = 0;
    for (uint32_t u = 0; u < U; u++) lsum += (uint64_t)(uint32_t)s->h_units[u].ltotal;
    if (lsum > 0xffffffffull) { delete s; return fail(ctx, GATB_ERR_RANGE, "sampler: more than 2^32 bases to place (uint32 counts would overflow)"); }

    {
        const char *why = nullptr;
        TRY(sampler_layout(s, st, &why));
        if (why) { delete s; return fail(ctx, GATB_ERR_INVALID, why); }
    }
    TRY(s->tally.alloc(3));
    TRY(s->unit_over.alloc(U));
    TRY(cudaStreamSynchronize(st));
#undef TRY
    if (e != cudaSuccess) { delete s; return fail(ctx, GATB_ERR_CUDA, cudaGetErrorString(e)); }
    if (ctx->trace)
        fprintf(stderr, "gatb_sampler_create: host checks %.2f ms, uploads + allocations queued %.2f, unit preparation done %.2f, layout done %.2f\n",
                t_host, t_uploads, t_prep, since());
    *out = s;
    return GATB_OK;
}

extern "C" void gatb_sampler_destroy(gatb_sampler *s)
{
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    delete s;
}

extern "C" uint64_t gatb_sampler_sample_capacity(const gatb_sampler *s) { return s ? s->placed_stride : 0; }

extern "C" int gatb_sampler_set_kind(gatb_sampler *s, int kind)
{
    if (!s) return GATB_ERR_INVALID;
    if (kind != 0 && kind != 1) return fail(s->ctx, GATB_ERR_INVALID, "sampler kind must be 0 (annotator) or 1 (segments)");
    // SamplerSegments returns unsorted, overlapping placements; only fromIsochores' merge(0) normalizes
    // them, and without it the reference's counters assert (gat/SegmentList.pyx:1032-1033)
    if (kind == 1 && !s->has_iso)
        return fail(s->ctx, GATB_ERR_INVALID, "SamplerSegments needs an isochore workspace: its samples are not normalized");
    if (s->no_hist)
        return fail(s->ctx, GATB_ERR_INVALID, "sampler was created without a length histogram (nbuckets = 0): SamplerShift only");
    s->kind = kind;
    return GATB_OK;
}

extern "C" int gatb_sampler_set_shift(gatb_sampler *s, double radius, int32_t extension)
{
    if (!s) return GATB_ERR_INVALID;
    gatb_ctx *ctx = s->ctx;
    if (!(radius >= 0.0) || radius > 1e6) return fail(ctx, GATB_ERR_INVALID, "SamplerShift: radius must be in [0, 1e6]");
    if (extension < 0) return fail(ctx, GATB_ERR_INVALID, "SamplerShift: extension must be >= 0");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    // A moved segment is cut at the gaps of the workspace inside its window: at most one piece per workspace
    // piece and fill, two fills per segment.  Room for eight pieces per segment (never more than that bound);
    // a unit that needs more reports GATB_ERR_CAPACITY instead of a wrong sample.
    for (uint32_t u = 0; u < s->n_units; u++) {
        UnitDesc &d = s->h_units[u];
        const uint64_t bound = 2ull * d.tab_n * ((uint64_t)d.ws_n + 1u);
        d.cap = next_pow2((uint32_t)std::min<uint64_t>(std::min<uint64_t>(bound, 8ull * d.tab_n + 256u) + 64u, 1u << 30));
    }
    const char *why = nullptr;
    cudaError_t e = sampler_layout(s, ctx->stream, &why);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail(ctx, GATB_ERR_CUDA, cudaGetErrorString(e));
    if (why) return fail(ctx, GATB_ERR_INVALID, why);
    s->kind = 2; s->shift_radius = radius; s->shift_extension = extension;
    return GATB_OK;
}

static uint32_t pick_batch(const gatb_sampler *s, uint64_t n_samples)
{
    uint64_t per_sample = (s->unit_stride + s->placed_stride) * 8 + (uint64_t)(s->n_units + s->n_contigs) * 5;
    uint64_t b = s->ctx->batch ? s->ctx->batch : 4096;
    const uint64_t limit = 24ull << 30;             // keep batch buffers under 24 GiB of the 180 GB HBM
    b = std::min<uint64_t>(b, std::max<uint64_t>(1, limit / std::max<uint64_t>(per_sample, 1)));
    b = std::min<uint64_t>(b, n_samples);
    return (uint32_t)std::max<uint64_t>(b, 1);
}

static int ensure_batch(gatb_sampler *s, uint32_t B)
{
    gatb_ctx *ctx = s->ctx;
    PlaceBufs &pb = ctx->scratch->pb;
    CU(ctx, pb.placed.ensure((uint64_t)B * s->placed_stride));
    CU(ctx, pb.placed_n.ensure((uint64_t)B * s->n_contigs));
    if (s->has_iso) {
        CU(ctx, pb.unit_buf.ensure((uint64_t)B * s->unit_stride));
        CU(ctx, pb.unit_n.ensure((uint64_t)B * s->n_units));
    }
    CU(ctx, pb.status.ensure((uint64_t)B * s->n_units));
    return GATB_OK;
}

__global__ void tally_kernel(const uint32_t *placed_n, uint64_t n_placed, const uint8_t *status, uint64_t n_status,
                             unsigned long long *tally)
{
    unsigned long long a = 0, r = 0, o = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_placed; i += (uint64_t)gridDim.x * blockDim.x)
        a += placed_n[i];
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_status; i += (uint64_t)gridDim.x * blockDim.x) {
        r += (status[i] & UNIT_HIT_ROUND_CAP) ? 1 : 0;
        o += (status[i] & UNIT_OVERFLOW) ? 1 : 0;
    }
    for (int d = 16; d > 0; d >>= 1) {
        a += __shfl_xor_sync(GATB_FULL, a, d);
        r += __shfl_xor_sync(GATB_FULL, r, d);
        o += __shfl_xor_sync(GATB_FULL, o, d);
    }
    if ((threadIdx.x & 31) == 0) {
        if (a) atomicAdd(&tally[0], a);
        if (r) atomicAdd(&tally[1], r);
        if (o) atomicAdd(&tally[2], o);
    }
}

// enqueue K1 (+K2) for one batch; result in s->placed / s->placed_n
static int place_batch(gatb_sampler *s, uint64_t seed, uint32_t track, uint64_t sample_begin, uint32_t B)
{
    gatb_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    PlaceBufs &pb = ctx->scratch->pb;
    PlaceParams p;
    memset(&p, 0, sizeof(p));
    p.units = s->units.p; p.order = s->order.p;
    p.ws_start = s->ws_start.p; p.ws_end = s->ws_end.p; p.ws_cuminc = s->ws_cuminc.p; p.len_tab = s->len_tab.p;
    p.ws_tab = s->ws_tab.p;
    if (s->has_iso) {
        p.buf = pb.unit_buf.p; p.sample_stride = s->unit_stride;
        p.out_n = pb.unit_n.p; p.out_n_stride = s->n_units; p.out_by_contig = 0;
    } else {
        p.buf = pb.placed.p; p.sample_stride = s->placed_stride;
        p.out_n = pb.placed_n.p; p.out_n_stride = s->n_contigs; p.out_by_contig = 1;
    }
    p.status = pb.status.p; p.unit_over = s->unit_over.p; p.n_units = s->n_units; p.one_piece = s->one_piece ? 1 : 0; p.n_samples = B; p.sample_begin = sample_begin;
    p.keys = philox_keys(seed); p.track = track; p.sampler_kind = s->kind;
    p.seg_start = s->seg_start.p; p.seg_end = s->seg_end.p;
    p.shift_half_radius = s->shift_radius / 2; p.shift_extension = s->shift_extension;
    { ProfScope ps(ctx, PROF_PLACE, st); launch_place(st, p); }
    CU(ctx, cudaGetLastError());
    if (s->has_iso) {
        MergeParams m;
        memset(&m, 0, sizeof(m));
        m.units = s->units.p; m.contig_unit_off = s->contig_unit_off.p; m.contig_units = s->contig_units.p;
        m.contig_base = s->contig_base.p; m.unit_buf = pb.unit_buf.p; m.unit_stride = s->unit_stride;
        m.unit_n = pb.unit_n.p; m.placed = pb.placed.p; m.placed_stride = s->placed_stride;
        m.placed_n = pb.placed_n.p; m.n_units = s->n_units; m.n_contigs = s->n_contigs; m.n_samples = B;
        { ProfScope ps(ctx, PROF_MERGE, st); launch_contig_merge(st, m); }
        CU(ctx, cudaGetLastError());
    }
    {
        ProfScope ps(ctx, PROF_OTHER, st);
        tally_kernel<<<std::min<uint32_t>(1024, (uint32_t)(((uint64_t)B * s->n_units + 255) / 256)), 256, 0, st>>>(
            pb.placed_n.p, (uint64_t)B * s->n_contigs, pb.status.p, (uint64_t)B * s->n_units, s->tally.p);
    }
    CU(ctx, cudaGetLastError());
    return GATB_OK;
}

// A unit that outgrew its buffer (UnitDesc.cap is an estimate, see prep_units_kernel): the reference and the
// oracle grow their lists on demand, so the call must not fail.  The flagged units get twice the room, the
// buffer layout is rebuilt and the caller runs the whole call again -- every draw is a function of (seed,
// track, unit, sample, turn), so the second pass reproduces the first one exactly, with room to finish.
// -> GATB_OK (grown; run again) or GATB_ERR_CAPACITY (a contig would need more than 2^24 slots).
static int grow_overflowed(gatb_sampler *s)
{
    gatb_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    std::vector<uint32_t> over(s->n_units);
    CU(ctx, cudaMemcpyAsync(over.data(), s->unit_over.p, s->n_units * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    bool any = false;
    for (uint32_t u = 0; u < s->n_units; u++)
        if (over[u]) {
            if (s->h_units[u].cap >= (1u << 24)) return fail(ctx, GATB_ERR_CAPACITY, "placement unit overflowed its segment buffer (2^24 slots)");
            s->h_units[u].cap *= 2u;
            any = true;
        }
    if (!any) return fail(ctx, GATB_ERR_CAPACITY, "placement unit overflowed its segment buffer");
    const char *why = nullptr;
    cudaError_t e = sampler_layout(s, st, &why);
    if (e != cudaSuccess) return fail(ctx, GATB_ERR_CUDA, cudaGetErrorString(e));
    if (why) return fail(ctx, GATB_ERR_CAPACITY, std::string("placement unit overflowed its segment buffer; ") + why);
    return GATB_OK;
}

static int check_place_args(gatb_sampler *s, uint32_t track, uint64_t sample_begin, uint64_t n_samples)
{
    gatb_ctx *ctx = s->ctx;
    if (sample_begin + n_samples > 0xffffffffull) return fail(ctx, GATB_ERR_RANGE, "sample index >= 2^32");
    if (track >= (1u << 24)) return fail(ctx, GATB_ERR_RANGE, "track index >= 2^24");
    if (s->no_hist && s->kind != 2)
        return fail(ctx, GATB_ERR_INVALID, "sampler was created without a length histogram (nbuckets = 0): call gatb_sampler_set_shift first");
    return GATB_OK;
}

// one pass of gatb_sampler_place / gatb_sampler_place_units; *overflowed: some unit needs a larger buffer
static int place_once(gatb_sampler *s, uint64_t seed, uint32_t track, uint64_t sample_begin, uint64_t n_samples,
                      bool by_unit, uint32_t *start, uint32_t *end, uint32_t *counts, uint64_t *base,
                      uint8_t *unit_status, bool *overflowed)
{
    gatb_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    PlaceBufs *sc = &ctx->scratch->pb;
    const bool from_units = by_unit && s->has_iso;          // the unit-level buffers (before fromIsochores)
    const uint64_t stride = from_units ? s->unit_stride : s->placed_stride;
    const uint32_t n_lists = by_unit ? s->n_units : s->n_contigs;
    std::vector<uint64_t> list_base(n_lists);
    for (uint32_t l = 0; l < n_lists; l++)
        list_base[l] = !by_unit ? s->h_contig_base[l] : from_units ? s->h_units[l].buf_off : s->h_contig_base[s->h_units[l].contig];
    if (base) for (uint32_t l = 0; l < n_lists; l++) base[l] = list_base[l];
    const uint32_t B = pick_batch(s, n_samples);
    int rc = ensure_batch(s, B);
    if (rc) return rc;
    CU(ctx, cudaMemsetAsync(s->tally.p, 0, 3 * sizeof(unsigned long long), st));
    CU(ctx, cudaMemsetAsync(s->unit_over.p, 0, s->n_units * sizeof(uint32_t), st));
    std::vector<uint64_t> h((uint64_t)B * stride);
    std::vector<uint32_t> hn((uint64_t)B * (from_units ? s->n_units : s->n_contigs));
    for (uint64_t done = 0; done < n_samples; done += B) {
        const uint32_t b = (uint32_t)std::min<uint64_t>(B, n_samples - done);
        rc = place_batch(s, seed, track, sample_begin + done, b);
        if (rc) return rc;
        CU(ctx, cudaMemcpyAsync(h.data(), from_units ? sc->unit_buf.p : sc->placed.p, (uint64_t)b * stride * 8, cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaMemcpyAsync(hn.data(), from_units ? sc->unit_n.p : sc->placed_n.p, (uint64_t)b * (from_units ? s->n_units : s->n_contigs) * 4,
                                cudaMemcpyDeviceToHost, st));
        if (unit_status)
            CU(ctx, cudaMemcpyAsync(unit_status + done * s->n_units, sc->status.p, (uint64_t)b * s->n_units, cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaStreamSynchronize(st));
        for (uint64_t sl = 0; sl < b; sl++)
            for (uint32_t l = 0; l < n_lists; l++) {
                const uint32_t n = (by_unit && !from_units) ? hn[sl * s->n_contigs + s->h_units[l].contig] : hn[sl * n_lists + l];
                counts[(done + sl) * n_lists + l] = n;
                const uint64_t src = sl * stride + list_base[l];
                const uint64_t dst = (done + sl) * stride + list_base[l];
                for (uint32_t i = 0; i < n; i++) { start[dst + i] = seg_start(h[src + i]); end[dst + i] = seg_end(h[src + i]); }
            }
    }
    unsigned long long tally[3];
    CU(ctx, cudaMemcpyAsync(tally, s->tally.p, sizeof(tally), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    *overflowed = tally[2] != 0;
    return GATB_OK;
}

static int place_impl(gatb_sampler *s, uint64_t seed, uint32_t track, uint64_t sample_begin, uint64_t n_samples,
                      bool by_unit, uint32_t *start, uint32_t *end, uint32_t *counts, uint64_t *base,
                      uint8_t *unit_status, uint64_t capacity)
{
    if (!s || !start || !end || !counts) return GATB_ERR_INVALID;
    gatb_ctx *ctx = s->ctx;
    int rc = check_place_args(s, track, sample_begin, n_samples);
    if (rc) return rc;
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    for (;;) {
        // the caller sized start/end from the capacity query: a grown layout may no longer fit them
        const uint64_t need = (by_unit && s->has_iso) ? s->unit_stride : s->placed_stride;
        if (capacity && need > capacity)
            return fail(ctx, GATB_ERR_CAPACITY, "placement buffers were grown: query the sample capacity again and repeat the call");
        bool overflowed = false;
        rc = place_once(s, seed, track, sample_begin, n_samples, by_unit, start, end, counts, base, unit_status, &overflowed);
        if (rc) return rc;
        if (!overflowed) return GATB_OK;
        rc = grow_overflowed(s);
        if (rc) return rc;
    }
}

extern "C" int gatb_sampler_place(gatb_sampler *s, uint64_t seed, uint32_t track, uint64_t sample_begin,
                                  uint64_t n_samples, uint32_t *start, uint32_t *end, uint32_t *counts,
                                  uint64_t *contig_base, uint8_t *unit_status)
{
    // (the arrays hold gatb_sampler_sample_capacity() slots per sample as queried BEFORE the call: a unit that
    // overflows grows the layout, which the fixed-size arrays cannot follow -> GATB_ERR_CAPACITY, query + repeat)
    const uint64_t cap = s ? s->placed_stride : 0;
    return place_impl(s, seed, track, sample_begin, n_samples, false, start, end, counts, contig_base, unit_status, cap);
}

extern "C" uint64_t gatb_sampler_unit_capacity(const gatb_sampler *s)
{
    return s ? (s->has_iso ? s->unit_stride : s->placed_stride) : 0;
}

extern "C" int gatb_sampler_place_units(gatb_sampler *s, uint64_t seed, uint32_t track, uint64_t sample_begin,
                                        uint64_t n_samples, uint32_t *start, uint32_t *end, uint32_t *counts,
                                        uint64_t *unit_base, uint8_t *unit_status)
{
    const uint64_t cap = s ? (s->has_iso ? s->unit_stride : s->placed_stride) : 0;
    return place_impl(s, seed, track, sample_begin, n_samples, true, start, end, counts, unit_base, unit_status, cap);
}

// one pass of gatb_run over all batches; tally[2] != 0: some unit needs a larger buffer (the counts are void)
static int run_once(gatb_sampler *s, const gatb_annotations *annos, int n_counters, const int32_t *counters,
                    uint64_t seed, uint32_t track, uint64_t sample_begin, uint64_t n_samples,
                    uint32_t *out_counts, double *out_density, int out_is_device, bool any_int, bool any_density,
                    unsigned long long *tally)
{
    gatb_ctx *ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    const uint32_t A = annos->n_annot;
    const uint32_t B = pick_batch(s, n_samples);
    const auto t_begin = std::chrono::steady_clock::now();
    auto since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
    double t_alloc = 0, t_placeq = 0, t_annos = 0, t_countq = 0;
    int rc = ensure_batch(s, B);
    if (rc) return rc;
    t_alloc = since();
    BatchScratch *sc = ctx->scratch;
    // Output routes, two ways to serve them (gatb_set_route_mode): (a) the counting kernel's epilogue stores every
    // row to every route itself (by_kernel = 1), (b) the kernel writes a plain staging slab and COPY ENGINES scatter
    // its rows / column blocks to the routes (2-D device-to-device copies on the copy stream, peer GPUs included)
    // while the compute stream goes on with the next batch -- the default: (a) put 7 x 16 MB of NVLink stores at the
    // very end of every 1.2 ms kernel, where nothing overlaps them (8 GPUs: 60.3 ms per step against 55.9 on one GPU).
    const bool routed = !ctx->routes.empty();
    const bool staged = !out_is_device || (routed && ctx->route_copy);
    const int n_stage = (staged && (n_samples > B || n_counters > 1)) ? 2 : 1;
    if (staged)
        for (int i = 0; i < n_stage; i++) {
            if (any_int) CU(ctx, sc->out_tmp[i].ensure((uint64_t)B * A));
            if (any_density && !out_is_device) CU(ctx, sc->out_tmp_f[i].ensure((uint64_t)B * A));
        }
    CU(ctx, cudaMemsetAsync(s->tally.p, 0, 3 * sizeof(unsigned long long), st));
    CU(ctx, cudaMemsetAsync(s->unit_over.p, 0, s->n_units * sizeof(uint32_t), st));
    // host outputs: the count kernels write a staging slab; its copy to the host runs on the copy stream while
    // the compute stream goes on with the next (counter, batch), which uses the other slab
    uint64_t n_staged = 0;
    bool copied_pending[2] = {false, false};
    for (uint64_t done = 0; done < n_samples; done += B) {
        const uint32_t b = (uint32_t)std::min<uint64_t>(B, n_samples - done);
        rc = place_batch(s, seed, track, sample_begin + done, b);
        if (rc) return rc;
        if (done == 0) t_placeq = since();
        CountParams p;
        memset(&p, 0, sizeof(p));
        p.placed = sc->pb.placed.p; p.sample_stride = s->placed_stride; p.key_base = s->contig_base.p;
        p.placed_n = sc->pb.placed_n.p; p.key_present = nullptr;
        for (int c = 0; c < n_counters; c++) {
            const bool dens = counters[c] == GATB_NUCLEOTIDE_DENSITY;
            rc = count_params_annos(annos, b, dens, p);
            if (rc) return rc;
            uint32_t *dst_u = out_counts ? out_counts + ((uint64_t)c * n_samples + done) * A : nullptr;
            double *dst_f = out_density ? out_density + done * A : nullptr;
            const int slab = (int)(n_staged % (uint64_t)n_stage);
            p.n_routes = 0;
            if (!dens && routed && !ctx->route_copy && out_is_device) {
                p.n_routes = (uint32_t)ctx->routes.size();
                for (uint32_t r = 0; r < p.n_routes; r++) {
                    const gatb_route &g = ctx->routes[r];
                    p.routes[r].base = g.base + (uint64_t)c * g.plane_stride;
                    p.routes[r].row_stride = g.row_stride;
                    p.routes[r].row0 = g.row0 + done;
                    p.routes[r].col_begin = g.col_begin; p.routes[r].col_end = std::min(g.col_end, A);
                }
            }
            const bool via_slab = !out_is_device || (routed && ctx->route_copy && !dens);
            p.out_u32 = via_slab ? sc->out_tmp[slab].p : dst_u;
            p.out_f64 = out_is_device ? dst_f : sc->out_tmp_f[slab].p;
            // annotations still uploading / building (gatb_annotations_create_async): the placement queued
            // above did not need them, the count does.  The host waits here (the GPU keeps placing) because
            // the build's outcome decides what may be launched: invalid lists or an index to rebuild.
            if (annos->pending) {
                rc = annotations_finish(const_cast<gatb_annotations *>(annos));
                tl_stream = ctx->stream;
                if (rc) { cudaStreamSynchronize(st); return rc; }
                t_annos = since();
            }
            if (via_slab && copied_pending[slab]) CU(ctx, cudaStreamWaitEvent(st, ctx->ev_copied[slab], 0));
            { ProfScope ps(ctx, PROF_COUNT); CU(ctx, launch_count(st, counters[c], p, ctx->count_threads)); }
            if (via_slab) {
                cudaStream_t cs = n_stage > 1 ? ctx->copy_stream : st;
                if (n_stage > 1) {
                    CU(ctx, cudaEventRecord(ctx->ev_counted[slab], st));
                    CU(ctx, cudaStreamWaitEvent(cs, ctx->ev_counted[slab], 0));
                }
                if (routed && !dens) {
                    // the rows of this batch to every route: columns [col_begin, col_end) of the slab -> the route's rows
                    for (const gatb_route &g : ctx->routes) {
                        const uint32_t ce = std::min(g.col_end, A);
                        if (ce <= g.col_begin) continue;
                        uint32_t *dst = g.base + (uint64_t)c * g.plane_stride + (g.row0 + done) * g.row_stride;
                        CU(ctx, cudaMemcpy2DAsync(dst, g.row_stride * sizeof(uint32_t), sc->out_tmp[slab].p + g.col_begin,
                                                  (size_t)A * sizeof(uint32_t), (size_t)(ce - g.col_begin) * sizeof(uint32_t), b,
                                                  cudaMemcpyDeviceToDevice, cs));
                    }
                }
                // host outputs (with routes as well: the rows go to the host AND to the routes)
                if (!out_is_device && dens) CU(ctx, cudaMemcpyAsync(dst_f, sc->out_tmp_f[slab].p, (uint64_t)b * A * sizeof(double), cudaMemcpyDeviceToHost, cs));
                else if (!out_is_device) CU(ctx, cudaMemcpyAsync(dst_u, sc->out_tmp[slab].p, (uint64_t)b * A * sizeof(uint32_t), cudaMemcpyDeviceToHost, cs));
                if (n_stage > 1) {
                    CU(ctx, cudaEventRecord(ctx->ev_copied[slab], cs));
                    copied_pending[slab] = true;
                }
                n_staged++;
            }
        }
    }
    // the compute stream joins the last copies: one synchronisation point for the caller
    for (int i = 0; i < 2; i++)
        if (copied_pending[i]) CU(ctx, cudaStreamWaitEvent(st, ctx->ev_copied[i], 0));
    t_countq = since();
    CU(ctx, cudaMemcpyAsync(tally, s->tally.p, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    if (ctx->trace)
        fprintf(stderr, "gatb_run: batch buffers %.2f ms, placement queued %.2f, annotations ready %.2f, all queued %.2f, done %.2f\n",
                t_alloc, t_placeq, t_annos, t_countq, since());
    return GATB_OK;
}

extern "C" int gatb_run(gatb_sampler *s, const gatb_annotations *annos, int n_counters, const int32_t *counters,
                        uint64_t seed, uint32_t track, uint64_t sample_begin, uint64_t n_samples,
                        uint32_t *out_counts, double *out_density, int out_is_device, uint64_t *info)
{
    if (!s || !annos || !counters || n_counters <= 0) return GATB_ERR_INVALID;
    gatb_ctx *ctx = s->ctx;
    if (annos->ctx != ctx) return fail(ctx, GATB_ERR_INVALID, "run: sampler and annotations belong to different contexts");
    if (annos->n_keys != s->n_contigs) return fail(ctx, GATB_ERR_INVALID, "run: annotations keys != sampler contigs");
    int rc = check_place_args(s, track, sample_begin, n_samples);
    if (rc) return rc;
    bool any_int = false, any_density = false;
    for (int c = 0; c < n_counters; c++) {
        if (counters[c] < 0 || counters[c] >= GATB_NCOUNTERS) return fail(ctx, GATB_ERR_INVALID, "unknown counter id");
        if (counters[c] == GATB_NUCLEOTIDE_DENSITY) any_density = true; else any_int = true;
    }
    if (any_density && (!annos->has_nseg || !out_density)) return fail(ctx, GATB_ERR_INVALID, "nucleotide-density needs key_ws_nseg and out_density");
    if (!ctx->routes.empty() && any_density)
        return fail(ctx, GATB_ERR_INVALID, "run: output routes deliver integer counters only");
    if (any_int && !out_counts && (ctx->routes.empty() || !out_is_device)) return fail(ctx, GATB_ERR_INVALID, "run: out_counts is NULL");
    if (n_samples == 0) return GATB_OK;
    if (!annos->pending && annos->status) return fail(ctx, annos->status, "run: the annotations failed validation");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    unsigned long long tally[3] = {0, 0, 0};
    for (;;) {
        rc = run_once(s, annos, n_counters, counters, seed, track, sample_begin, n_samples, out_counts, out_density,
                      out_is_device, any_int, any_density, tally);
        if (rc) return rc;
        if (tally[2] == 0) break;
        rc = grow_overflowed(s);            // (rare: skewed units, see prep_units_kernel) then the call runs again
        if (rc) return rc;
    }
    if (info) { info[0] = tally[0]; info[1] = tally[1]; info[2] = tally[2]; }
    rc = annotations_finish(const_cast<gatb_annotations *>(annos));      // invalid lists: the counts mean nothing
    if (rc) return rc;
    return GATB_OK;
}

// work of the counting kernel on the LAST batch of the preceding gatb_run on this sampler (its placed segments
// are still in the context's batch buffers): out[0] = segments, out[1] = index entries in their runs (what the
// kernel tests, padding included), out[2] = entries of the whole index, out[3] = bytes of the index arrays the
// kernel reads (offsets + entries)
extern "C" int gatb_count_work(gatb_sampler *s, const gatb_annotations *annos, uint32_t n_samples, uint64_t *out)
{
    if (!s || !annos || !out) return GATB_ERR_INVALID;
    gatb_ctx *ctx = s->ctx;
    if (annos->ctx != ctx || annos->n_keys != s->n_contigs) return fail(ctx, GATB_ERR_INVALID, "count_work: sampler / annotations mismatch");
    CU(ctx, cudaSetDevice(ctx->device));
    int rc = annotations_finish(const_cast<gatb_annotations *>(annos));
    if (rc) return rc;
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    if (ctx->scratch->pb.placed.n < (uint64_t)n_samples * s->placed_stride || ctx->scratch->pb.placed_n.n < (uint64_t)n_samples * s->n_contigs)
        return fail(ctx, GATB_ERR_INVALID, "count_work: no batch of that size has been placed");
    CountParams p;
    memset(&p, 0, sizeof(p));
    rc = count_params_annos(annos, n_samples, false, p);
    if (rc) return rc;
    p.placed = ctx->scratch->pb.placed.p; p.sample_stride = s->placed_stride; p.key_base = s->contig_base.p;
    p.placed_n = ctx->scratch->pb.placed_n.p;
    DevBuf<unsigned long long> d_out;
    CU(ctx, d_out.alloc(2));
    CU(ctx, cudaMemsetAsync(d_out.p, 0, 2 * sizeof(unsigned long long), st));
    { ProfScope ps(ctx, PROF_OTHER); launch_count_work(st, p, d_out.p); }
    CU(ctx, cudaGetLastError());
    unsigned long long h[2];
    CU(ctx, cudaMemcpyAsync(h, d_out.p, sizeof(h), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    out[0] = h[0]; out[1] = h[1];
    out[2] = annos->n_entries;
    out[3] = annos->n_boff * sizeof(uint4) + annos->n_entries * sizeof(uint2);
    return GATB_OK;
}

// ---------------------------------------------------------------------------------------------------
// column statistics
// getTwoSidedPValue (gat/Engine.pyx:1543-1576): the index of two_sided_index (count.cuh), divided by l
static double two_sided_pvalue(uint64_t l, uint64_t n_lt, uint64_t n_eq, double value, double centre)
{
    return std::max(1.0 / (double)l, (double)two_sided_index(l, n_lt, n_eq, value, centre) / (double)l);
}

// The per-column doubles of makeEnrichmentStatistics (gat/Engine.pyx:1635-1718) from a column's reduced integers /
// order statistics: ONE function for the matrix (gatb_column_stats) and the matrix-free path (gatb_colacc_finish),
// so that both produce their doubles from the same numbers by the same operations.  mean = sum / l, sumsq = sum
// (x - mean)^2, qlo / qhi the order statistics at the CI ranks, n_lt / n_eq the counts of pass 1 against obs_eff
// (= observed / ref_fold).  Any output may be NULL.
static void finish_columns(uint64_t l, uint32_t A, const double *observed, const double *obs_eff, const double *ref_fold,
                           double pseudo_count, const double *mean, const double *sumsq, const double *qlo,
                           const double *qhi, const unsigned long long *n_lt, const unsigned long long *n_eq,
                           double *expected, double *stddev, double *lower95, double *upper95, double *fold, double *pvalue)
{
    for (uint32_t a = 0; a < A; a++) {
        double exp_ = mean[a];
        if (ref_fold) exp_ *= ref_fold[a];                                    // :1673-1676
        const double fo = (exp_ != 0) ? (observed[a] + pseudo_count) / (exp_ + pseudo_count) : 1.0;   // :1679-1682
        double lo = qlo[a], hi = qhi[a];
        if (ref_fold) { lo *= ref_fold[a]; hi *= ref_fold[a]; }              // :1713-1714
        if (expected) expected[a] = exp_;
        if (stddev) stddev[a] = std::sqrt(sumsq[a] / (double)l);             // numpy.std ddof 0 (:1684)
        if (lower95) lower95[a] = lo;
        if (upper95) upper95[a] = hi;
        if (fold) fold[a] = fo;
        if (pvalue) pvalue[a] = two_sided_pvalue(l, n_lt[a], n_eq[a], obs_eff[a], exp_);
    }
}

// observed / ref_fold (the value the samples are compared with) and the CI ranks (gat/Engine.pyx:1689-1696)
static int effective_observed(gatb_ctx *ctx, uint32_t A, const double *observed, const double *ref_fold, std::vector<double> &obs_eff)
{
    obs_eff.resize(A);
    for (uint32_t a = 0; a < A; a++) {
        if (ref_fold) {
            if (!(ref_fold[a] > 0)) return fail(ctx, GATB_ERR_INVALID, "0 fold change not applicable");
            obs_eff[a] = observed[a] / ref_fold[a];
        } else obs_eff[a] = observed[a];
    }
    return GATB_OK;
}
static void ci_ranks(uint64_t l, uint64_t &rank_lo, uint64_t &rank_hi)
{
    const uint64_t off = (uint64_t)(0.05 * (double)l);
    if (off > 0) { rank_lo = std::min<uint64_t>(off, l - 1); rank_hi = (l > off) ? l - off : 0; }
    else { rank_lo = 0; rank_hi = l - 1; }
}

// the context's device and stream for a statistics call, and its input matrix on the device: the caller's own, or a
// copy of the host one held by `copy`
static int device_matrix(gatb_ctx *ctx, const void *counts, int is_float, int counts_is_device, uint64_t n,
                         DevBuf<uint8_t> &copy, const void *&dc)
{
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    dc = counts;
    if (counts_is_device) return GATB_OK;
    CU(ctx, copy.upload((const uint8_t *)counts, n * (is_float ? sizeof(double) : sizeof(uint32_t)), ctx->stream));
    dc = copy.p;
    return GATB_OK;
}

// The exact integers of statistics pass 1 over a uint32 counter plane (gatb_column_stats, gatb_column_pvalue, the column
// accumulator): every kernel that counts rows ADDS its integers here, so any split of the rows and any choice of kernel
// gives the same integers, and finish_columns() the same doubles.
struct ColumnSums {
    enum { ISUM, N_LT, N_EQ, SQ_LO, SQ_HI, N_INTS };   // sum, #{x < obs_eff}, #{x == obs_eff}, 128-bit sum of squares
    gatb_ctx *ctx = nullptr;
    uint32_t A = 0;
    std::vector<double> obs_eff;
    std::vector<uint32_t> h_thr;                    // lt_thr | eq_val | flags: obs_eff as integer tests (streamed pass 1)
    DevBuf<uint32_t> thr;
    DevBuf<double> d_obs;                           // obs_eff (column-tiled pass 1)
    DevBuf<unsigned long long> ints;                // [N_INTS][A]: gatb_colacc_state's `moments`
    DevBuf<uint32_t> mm;                            // min | max [2][A], then vmax, error (a TMA copy did not complete)
    std::vector<unsigned long long> h_ints;         // host copies (fetch)
    std::vector<uint32_t> h_mm;
    uint64_t rows = 0;                              // rows counted so far
    bool streamed = false;                          // the last add took the streamed pass (and vmax is the matrix maximum)
    unsigned long long *dev(int k) { return ints.p + (size_t)k * A; }
    const unsigned long long *host(int k) const { return h_ints.data() + (size_t)k * A; }
    uint32_t *error() { return mm.p + 2 * (size_t)A + 1; }
    uint32_t vmax() const { return h_mm[2 * (size_t)A]; }
    int init(gatb_ctx *c, uint32_t n_cols, const double *observed, const double *ref_fold)
    {
        ctx = c; A = n_cols;
        if (const int rc = effective_observed(ctx, A, observed, ref_fold, obs_eff)) return rc;
        cudaStream_t st = ctx->stream;
        h_thr.resize(3 * (size_t)A);
        stats_stream_thresholds(obs_eff.data(), A, h_thr.data(), h_thr.data() + A, h_thr.data() + 2 * (size_t)A);
        h_mm.assign(2 * (size_t)A + 2, 0u);
        std::fill(h_mm.begin(), h_mm.begin() + A, 0xffffffffu);
        CU(ctx, thr.upload(h_thr.data(), h_thr.size(), st));
        CU(ctx, d_obs.upload(obs_eff.data(), A, st));
        CU(ctx, ints.alloc(N_INTS * (size_t)A));
        CU(ctx, cudaMemsetAsync(ints.p, 0, N_INTS * (size_t)A * sizeof(unsigned long long), st));
        CU(ctx, mm.upload(h_mm.data(), h_mm.size(), st));
        return GATB_OK;
    }
    // counts the first A values of n_rows rows, row_stride apart, into the sums (`extremes`: into min | max as well).
    // The TMA-streamed pass of stats_stream.cu unless GATB_STATS_STREAM=0 or the rows are strided, wider than a ring
    // stage or not 4-byte aligned; then the column-tiled pass of count.cu
    int add(const uint32_t *counts, uint64_t n_rows, uint64_t row_stride, bool extremes)
    {
        cudaStream_t st = ctx->stream;
        streamed = row_stride == A && ctx->stats_stream && stats_stream_fits(counts, n_rows, A, ctx->smem_optin);
        if (streamed) {
            StreamStatsParams p;
            memset(&p, 0, sizeof(p));
            p.counts = counts; p.n_samples = n_rows; p.n_cols = A;
            stats_stream_geometry(p);
            p.lt_thr = thr.p; p.eq_val = thr.p + A; p.col_flags = thr.p + 2 * (size_t)A;
            p.isum = dev(ISUM); p.n_lt = dev(N_LT); p.n_eq = dev(N_EQ); p.sq_lo = dev(SQ_LO); p.sq_hi = dev(SQ_HI);
            if (extremes) { p.col_min = mm.p; p.col_max = mm.p + A; }
            p.vmax = mm.p + 2 * (size_t)A; p.error = error();
            ProfScope ps(ctx, PROF_OTHER);
            CU(ctx, launch_stats_stream_pass1(st, p, ctx->sm_count));
        } else {
            StatsParams p;
            memset(&p, 0, sizeof(p));
            p.counts = counts; p.n_samples = n_rows; p.n_cols = A; p.row_stride = row_stride; p.observed = d_obs.p;
            p.isum = dev(ISUM); p.n_lt = dev(N_LT); p.n_eq = dev(N_EQ); p.sq_lo = dev(SQ_LO); p.sq_hi = dev(SQ_HI);
            if (extremes) { p.col_min = mm.p; p.col_max = mm.p + A; }
            ProfScope ps(ctx, PROF_OTHER);
            launch_stats_pass1(st, p);
            CU(ctx, cudaGetLastError());
        }
        rows += n_rows;
        return GATB_OK;
    }
    // the integers and min | max | vmax to h_ints / h_mm, with the stream drained
    int fetch()
    {
        cudaStream_t st = ctx->stream;
        h_ints.resize(N_INTS * (size_t)A);
        CU(ctx, cudaMemcpyAsync(h_ints.data(), ints.p, h_ints.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaMemcpyAsync(h_mm.data(), mm.p, h_mm.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaStreamSynchronize(st));
        if (h_mm[2 * (size_t)A + 1]) return fail(ctx, GATB_ERR_CUDA, "column statistics: a TMA copy did not complete");
        return GATB_OK;
    }
    // once the sums hold all l samples of every column: mean = sum / l and sumsq = sum (x - mean)^2 = (l * sum x^2 -
    // (sum x)^2) / l with the numerator exact in 128 bits (x < 2^32, l < 2^32: both products stay below 2^128), rounded
    // once when it becomes a double; host(N_LT), host(N_EQ) and vmax() hold the rest
    int read(uint64_t l, std::vector<double> &mean, std::vector<double> &sumsq)
    {
        if (const int rc = fetch()) return rc;
        mean.resize(A); sumsq.resize(A);
        for (uint32_t a = 0; a < A; a++) {
            const unsigned long long sum = host(ISUM)[a];
            const unsigned __int128 sq = ((unsigned __int128)host(SQ_HI)[a] << 64) | host(SQ_LO)[a];
            mean[a] = (double)sum / (double)l;                              // numpy.mean (:1671)
            sumsq[a] = (double)((unsigned __int128)l * sq - (unsigned __int128)sum * sum) / (double)l;
        }
        return GATB_OK;
    }
    // adds another state (gatb_colacc_state layout; either part may be NULL) into this one: the sums of its n_rows rows
    // with the carry into the high word of the sum of squares, the extremes folded
    int merge(uint64_t n_rows, const uint64_t *ints_in, const uint32_t *minmax)
    {
        if (const int rc = fetch()) return rc;
        cudaStream_t st = ctx->stream;
        const size_t n = A;
        if (ints_in) {
            for (size_t a = 0; a < n; a++) {
                unsigned long long *m = h_ints.data() + a;
                const uint64_t *o = ints_in + a;
                const unsigned __int128 z = (((unsigned __int128)m[SQ_HI * n] << 64) | m[SQ_LO * n]) +
                                            (((unsigned __int128)o[SQ_HI * n] << 64) | o[SQ_LO * n]);
                m[SQ_LO * n] = (uint64_t)z; m[SQ_HI * n] = (uint64_t)(z >> 64);
                for (const size_t k : {ISUM, N_LT, N_EQ}) m[k * n] += o[k * n];
            }
            CU(ctx, cudaMemcpyAsync(ints.p, h_ints.data(), h_ints.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
            rows += n_rows;
        }
        if (minmax) {
            for (size_t a = 0; a < n; a++) { h_mm[a] = std::min(h_mm[a], minmax[a]); h_mm[n + a] = std::max(h_mm[n + a], minmax[n + a]); }
            CU(ctx, cudaMemcpyAsync(mm.p, h_mm.data(), 2 * n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        }
        return GATB_OK;
    }
};

// q = the values at ranks[0] | ranks[1] of every column of the uint32 matrix [l][A] that `sums` has counted: the streamed
// radix select (4 bits per pass from the top nibble of the matrix maximum) where pass 1 was streamed, else the tiled one
static int order_stats_u32(ColumnSums &sums, const uint32_t *dc, uint64_t l, const uint64_t *ranks, std::vector<double> &q)
{
    gatb_ctx *ctx = sums.ctx;
    const uint32_t A = sums.A;
    cudaStream_t st = ctx->stream;
    DevBuf<double> d_q;
    CU(ctx, d_q.alloc(2 * (size_t)A));
    DevBuf<unsigned long long> d_rank;              // rank | rank_out
    DevBuf<uint32_t> d_prefix, d_hist;              // prefix | prefix_out
    std::vector<unsigned long long> h_rank(4 * (size_t)A, ranks[1]);
    if (sums.streamed) {
        std::fill_n(h_rank.begin(), A, ranks[0]);
        CU(ctx, d_rank.upload(h_rank.data(), h_rank.size(), st));
        CU(ctx, d_prefix.alloc(4 * (size_t)A));
        CU(ctx, cudaMemsetAsync(d_prefix.p, 0, 4 * (size_t)A * sizeof(uint32_t), st));
        CU(ctx, d_hist.alloc(32 * (size_t)A));
        CU(ctx, cudaMemsetAsync(d_hist.p, 0, 32 * (size_t)A * sizeof(uint32_t), st));
        StreamStatsParams p;
        memset(&p, 0, sizeof(p));
        p.counts = dc; p.n_samples = l; p.n_cols = A;
        stats_stream_geometry(p);
        p.prefix = d_prefix.p; p.prefix_out = d_prefix.p + 2 * (size_t)A;
        p.rank = d_rank.p; p.rank_out = d_rank.p + 2 * (size_t)A;
        p.hist = d_hist.p; p.q_lo = d_q.p; p.q_hi = d_q.p + A; p.error = sums.error();
        int top = 0;
        while (top < 28 && (sums.vmax() >> (top + 4)) != 0u) top += 4;
        for (int shift = top; shift >= 0; shift -= 4) {
            p.shift = (uint32_t)shift;
            ProfScope ps(ctx, PROF_OTHER);
            CU(ctx, launch_stats_stream_select(st, p, ctx->sm_count, ctx->smem_optin));
        }
    } else {
        StatsParams p;
        memset(&p, 0, sizeof(p));
        p.counts = dc; p.n_samples = l; p.n_cols = A;
        p.q_lo = d_q.p; p.q_hi = d_q.p + A; p.rank_lo = ranks[0]; p.rank_hi = ranks[1];
        { ProfScope ps(ctx, PROF_OTHER); launch_stats_select(st, p); }
        CU(ctx, cudaGetLastError());
    }
    q.resize(2 * (size_t)A);
    CU(ctx, cudaMemcpyAsync(q.data(), d_q.p, q.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    return sums.fetch();                            // (synchronises; fails if a copy of a select pass did not complete)
}

// float64 matrices (nucleotide-density, gat-compare) keep the column-tiled kernels of count.cu.  Pass 1: cnt = n_lt |
// n_eq against obs and the column means; with `ranks`, pass 2 for sum (x - mean)^2 and the 8-bit radix select for
// q = the values at ranks[0] | ranks[1]
static int float_stats(gatb_ctx *ctx, const double *dc, uint64_t l, uint32_t A, const double *obs, const uint64_t *ranks,
                       std::vector<unsigned long long> &cnt, std::vector<double> &mean, std::vector<double> &sumsq,
                       std::vector<double> &q)
{
    cudaStream_t st = ctx->stream;
    DevBuf<double> d_obs, d_sum, d_mean, d_sq, d_q;
    DevBuf<unsigned long long> d_cnt;
    CU(ctx, d_obs.upload(obs, A, st));
    CU(ctx, d_sum.alloc(A));
    CU(ctx, d_cnt.alloc(2 * (size_t)A));
    StatsParams p;
    memset(&p, 0, sizeof(p));
    p.counts = dc; p.is_float = 1; p.n_samples = l; p.n_cols = A; p.observed = d_obs.p;
    p.sum = d_sum.p; p.n_lt = d_cnt.p; p.n_eq = d_cnt.p + A;
    { ProfScope ps(ctx, PROF_OTHER); launch_stats_pass1(st, p); }
    CU(ctx, cudaGetLastError());
    cnt.resize(2 * (size_t)A); mean.resize(A);
    CU(ctx, cudaMemcpyAsync(cnt.data(), d_cnt.p, cnt.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaMemcpyAsync(mean.data(), d_sum.p, A * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    for (uint32_t a = 0; a < A; a++) mean[a] /= (double)l;                  // numpy.mean (:1671)
    if (!ranks) return GATB_OK;
    CU(ctx, d_mean.upload(mean.data(), A, st));
    CU(ctx, d_sq.alloc(A)); CU(ctx, d_q.alloc(2 * (size_t)A));
    p.mean = d_mean.p; p.sumsq_dev = d_sq.p; p.q_lo = d_q.p; p.q_hi = d_q.p + A; p.rank_lo = ranks[0]; p.rank_hi = ranks[1];
    { ProfScope ps(ctx, PROF_OTHER); launch_stats_pass2(st, p); }
    { ProfScope ps(ctx, PROF_OTHER); launch_stats_select(st, p); }
    CU(ctx, cudaGetLastError());
    sumsq.resize(A); q.resize(2 * (size_t)A);
    CU(ctx, cudaMemcpyAsync(sumsq.data(), d_sq.p, A * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaMemcpyAsync(q.data(), d_q.p, q.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    return GATB_OK;
}

extern "C" int gatb_column_stats(gatb_ctx *ctx, const void *counts, int is_float, int counts_is_device,
                                 uint64_t n_samples, int n_cols, const double *observed, const double *ref_fold,
                                 double pseudo_count, double *expected, double *stddev, double *lower95,
                                 double *upper95, double *fold, double *pvalue)
{
    if (!ctx || !counts || !observed || n_cols <= 0) return GATB_ERR_INVALID;
    if (n_samples < 1) return fail(ctx, GATB_ERR_INVALID, "column_stats: no samples");
    const uint32_t A = (uint32_t)n_cols;
    const uint64_t l = n_samples;
    DevBuf<uint8_t> d_counts;
    const void *dc = nullptr;
    int rc = device_matrix(ctx, counts, is_float, counts_is_device, l * A, d_counts, dc);
    if (rc) return rc;
    uint64_t ranks[2];
    ci_ranks(l, ranks[0], ranks[1]);
    ColumnSums sums;
    std::vector<double> obs_eff, mean, sumsq, q;
    std::vector<unsigned long long> cnt;            // float64: n_lt | n_eq
    const unsigned long long *n_lt, *n_eq;
    if (!is_float) {
        rc = sums.init(ctx, A, observed, ref_fold);
        if (!rc) rc = sums.add((const uint32_t *)dc, l, A, false);
        if (!rc) rc = sums.read(l, mean, sumsq);
        if (!rc) rc = order_stats_u32(sums, (const uint32_t *)dc, l, ranks, q);
        obs_eff = sums.obs_eff; n_lt = sums.host(ColumnSums::N_LT); n_eq = sums.host(ColumnSums::N_EQ);
    } else {
        rc = effective_observed(ctx, A, observed, ref_fold, obs_eff);
        if (!rc) rc = float_stats(ctx, (const double *)dc, l, A, obs_eff.data(), ranks, cnt, mean, sumsq, q);
        n_lt = cnt.data(); n_eq = cnt.data() + A;
    }
    if (rc) return rc;
    finish_columns(l, A, observed, obs_eff.data(), ref_fold, pseudo_count, mean.data(), sumsq.data(), q.data(), q.data() + A,
                   n_lt, n_eq, expected, stddev, lower95, upper95, fold, pvalue);
    return GATB_OK;
}

// empirical p-value of values[a] in column a given the column's STORED expectation
// (AnnotatorResult.getEmpiricalPValue -> getTwoSidedPValue(&self.stats, value), gat/Engine.pyx:1543-1576, :1829-1831):
// the over / under-representation branch compares with stats.expected (already multiplied by a reference
// fold, :1673-1676), not with a recomputed sample mean
extern "C" int gatb_column_pvalue(gatb_ctx *ctx, const void *counts, int is_float, int counts_is_device,
                                  uint64_t n_samples, int n_cols, const double *values, const double *expected,
                                  double *pvalue)
{
    if (!ctx || !counts || !values || !expected || !pvalue || n_cols <= 0) return GATB_ERR_INVALID;
    if (n_samples < 1) return fail(ctx, GATB_ERR_INVALID, "column_pvalue: no samples");
    const uint32_t A = (uint32_t)n_cols;
    const uint64_t l = n_samples;
    DevBuf<uint8_t> d_counts;
    const void *dc = nullptr;
    int rc = device_matrix(ctx, counts, is_float, counts_is_device, l * A, d_counts, dc);
    if (rc) return rc;
    ColumnSums sums;
    std::vector<double> mean, sumsq, unused;
    std::vector<unsigned long long> cnt;            // float64: n_lt | n_eq
    const unsigned long long *n_lt, *n_eq;
    if (!is_float) {
        rc = sums.init(ctx, A, values, nullptr);
        if (!rc) rc = sums.add((const uint32_t *)dc, l, A, false);
        if (!rc) rc = sums.read(l, mean, sumsq);
        n_lt = sums.host(ColumnSums::N_LT); n_eq = sums.host(ColumnSums::N_EQ);
    } else {
        rc = float_stats(ctx, (const double *)dc, l, A, values, nullptr, cnt, mean, unused, unused);
        n_lt = cnt.data(); n_eq = cnt.data() + A;
    }
    if (rc) return rc;
    for (uint32_t a = 0; a < A; a++) pvalue[a] = two_sided_pvalue(l, n_lt[a], n_eq[a], values[a], expected[a]);
    return GATB_OK;
}

// ---------------------------------------------------------------------------------------------------
// column statistics without the sample matrix: an accumulator of one uint32 counter plane, fed slab by slab.
// Pass 1 of the statistics ADDS its exact integers into the accumulator's ColumnSums, so any split of the rows into
// slabs gives the integers of one pass over the whole matrix; the two order statistics come from per-column windows
// of unit-width bins (exact values, so exact ranks).  gatb_colacc_finish turns the integers into doubles with the
// same finish_columns() as gatb_column_stats: same integers, same doubles.
struct gatb_colacc {
    gatb_ctx *ctx = nullptr;
    uint32_t A = 0;
    uint64_t l = 0;                                 // samples of the whole column
    std::vector<double> observed, ref;
    ColumnSums sums;
    uint64_t n_bins = 0;
    DevBuf<unsigned long long> outside;             // below | above [2][A]
    DevBuf<uint32_t> win;                           // lo | width [2][A]
    DevBuf<unsigned long long> bin_off;             // [A]
    DevBuf<uint32_t> bins;                          // [n_bins]
};

extern "C" int gatb_colacc_create(gatb_ctx *ctx, int n_cols, uint64_t n_samples_total, const double *observed,
                                  const double *ref_fold, gatb_colacc **out)
{
    if (!ctx || !observed || !out || n_cols <= 0) return GATB_ERR_INVALID;
    *out = nullptr;
    if (n_samples_total < 1 || n_samples_total >= (1ull << 32))
        return fail(ctx, GATB_ERR_INVALID, "colacc_create: n_samples_total must be in [1, 2^32)");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    std::unique_ptr<gatb_colacc> c(new gatb_colacc());
    c->ctx = ctx; c->A = (uint32_t)n_cols; c->l = n_samples_total;
    const uint32_t A = c->A;
    c->observed.assign(observed, observed + A);
    if (ref_fold) c->ref.assign(ref_fold, ref_fold + A);
    if (const int rc = c->sums.init(ctx, A, observed, ref_fold)) return rc;
    CU(ctx, c->outside.alloc(2 * (size_t)A));
    CU(ctx, cudaMemsetAsync(c->outside.p, 0, 2 * (size_t)A * sizeof(unsigned long long), st));
    CU(ctx, c->win.alloc(2 * (size_t)A));
    CU(ctx, cudaMemsetAsync(c->win.p, 0, 2 * (size_t)A * sizeof(uint32_t), st));
    CU(ctx, c->bin_off.alloc(A));
    CU(ctx, cudaMemsetAsync(c->bin_off.p, 0, A * sizeof(unsigned long long), st));
    *out = c.release();
    return GATB_OK;
}

extern "C" int gatb_colacc_set_windows(gatb_colacc *c, const uint32_t *lo, const uint32_t *width)
{
    if (!c || !lo || !width) return GATB_ERR_INVALID;
    gatb_ctx *ctx = c->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    const uint32_t A = c->A;
    std::vector<unsigned long long> h_off(A);
    uint64_t n = 0;
    for (uint32_t a = 0; a < A; a++) {
        if ((uint64_t)lo[a] + width[a] > (1ull << 32)) return fail(ctx, GATB_ERR_INVALID, "colacc_set_windows: window past 2^32");
        h_off[a] = n;
        n += width[a];
    }
    CU(ctx, c->bins.alloc(std::max<uint64_t>(n, 1)));
    c->n_bins = n;
    CU(ctx, cudaMemsetAsync(c->bins.p, 0, std::max<uint64_t>(n, 1) * sizeof(uint32_t), st));
    CU(ctx, cudaMemsetAsync(c->outside.p, 0, 2 * (size_t)A * sizeof(unsigned long long), st));
    CU(ctx, cudaMemcpyAsync(c->win.p, lo, A * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    CU(ctx, cudaMemcpyAsync(c->win.p + A, width, A * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    CU(ctx, cudaMemcpyAsync(c->bin_off.p, h_off.data(), A * sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
    CU(ctx, cudaStreamSynchronize(st));
    return GATB_OK;
}

extern "C" int gatb_colacc_add(gatb_colacc *c, const uint32_t *counts, uint64_t n_rows, uint64_t row_stride, int what)
{
    if (!c) return GATB_ERR_INVALID;
    gatb_ctx *ctx = c->ctx;
    const uint32_t A = c->A;
    if (what & ~(GATB_COLACC_SUMS | GATB_COLACC_HIST)) return fail(ctx, GATB_ERR_INVALID, "colacc_add: unknown flags");
    if (n_rows == 0) return GATB_OK;
    if (!counts || row_stride < A) return fail(ctx, GATB_ERR_INVALID, "colacc_add: no slab or row_stride < n_cols");
    if ((what & GATB_COLACC_SUMS) && c->sums.rows + n_rows > c->l)
        return fail(ctx, GATB_ERR_INVALID, "colacc_add: more rows than n_samples_total");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    if (what & GATB_COLACC_SUMS)
        if (const int rc = c->sums.add(counts, n_rows, row_stride, true)) return rc;
    if (what & GATB_COLACC_HIST) {
        ColHistParams h;
        memset(&h, 0, sizeof(h));
        h.counts = counts; h.n_rows = n_rows; h.row_stride = row_stride; h.n_cols = A;
        h.lo = c->win.p; h.width = c->win.p + A; h.bin_off = c->bin_off.p; h.bins = c->bins.p; h.outside = c->outside.p;
        ProfScope ps(ctx, PROF_OTHER);
        CU(ctx, launch_colacc_hist(ctx->stream, h, ctx->sm_count));
    }
    return GATB_OK;
}

extern "C" int gatb_colacc_state(gatb_colacc *c, uint64_t *rows, uint64_t *moments, uint32_t *minmax, uint64_t *outside,
                                 uint32_t *bins)
{
    if (!c) return GATB_ERR_INVALID;
    gatb_ctx *ctx = c->ctx;
    const size_t A = c->A;
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    if (const int rc = c->sums.fetch()) return rc;
    if (rows) *rows = c->sums.rows;
    if (moments) std::copy(c->sums.h_ints.begin(), c->sums.h_ints.end(), moments);
    if (minmax) std::copy(c->sums.h_mm.begin(), c->sums.h_mm.begin() + 2 * A, minmax);
    if (outside) CU(ctx, cudaMemcpyAsync(outside, c->outside.p, 2 * A * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (bins && c->n_bins) CU(ctx, cudaMemcpyAsync(bins, c->bins.p, c->n_bins * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    return GATB_OK;
}

extern "C" int gatb_colacc_merge(gatb_colacc *c, uint64_t rows, const uint64_t *moments, const uint32_t *minmax,
                                 const uint64_t *outside, const uint32_t *bins)
{
    if (!c) return GATB_ERR_INVALID;
    gatb_ctx *ctx = c->ctx;
    const size_t A = c->A;
    if (c->sums.rows + rows > c->l) return fail(ctx, GATB_ERR_INVALID, "colacc_merge: more rows than n_samples_total");
    // (only the parts given come down to the host: a merge of the sums alone does not move the arena)
    std::vector<uint64_t> o(outside ? 2 * A : 0);
    std::vector<uint32_t> b(bins ? c->n_bins : 0);
    if (const int rc = gatb_colacc_state(c, nullptr, nullptr, nullptr, outside ? o.data() : nullptr,
                                         bins ? b.data() : nullptr)) return rc;
    if (const int rc = c->sums.merge(rows, moments, minmax)) return rc;
    cudaStream_t st = ctx->stream;
    if (outside) {
        for (size_t i = 0; i < 2 * A; i++) o[i] += outside[i];
        CU(ctx, cudaMemcpyAsync(c->outside.p, o.data(), 2 * A * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    }
    if (bins && c->n_bins) {
        for (uint64_t i = 0; i < c->n_bins; i++) b[i] += bins[i];
        CU(ctx, cudaMemcpyAsync(c->bins.p, b.data(), c->n_bins * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    }
    CU(ctx, cudaStreamSynchronize(st));
    return GATB_OK;
}

static ColSparseParams sparse_params(gatb_colacc *c)
{
    ColSparseParams p;
    memset(&p, 0, sizeof(p));
    p.n_cols = c->A; p.lo = c->win.p; p.width = c->win.p + c->A; p.bin_off = c->bin_off.p; p.bins = c->bins.p;
    return p;
}

// the windows' non-zero bins as CSR, compacted on the device: only the sparse arrays come to the host
extern "C" int gatb_colacc_export(gatb_colacc *c, int64_t *col_ptr, uint32_t *value, uint64_t *count, uint64_t capacity)
{
    if (!c || !col_ptr || (!value) != (!count)) return GATB_ERR_INVALID;
    gatb_ctx *ctx = c->ctx;
    const uint32_t A = c->A;
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    ColSparseParams p = sparse_params(c);
    DevBuf<unsigned long long> d_nnz;
    CU(ctx, d_nnz.alloc(A));
    p.nnz = d_nnz.p;
    { ProfScope ps(ctx, PROF_OTHER); CU(ctx, launch_colacc_export(st, p, false)); }
    std::vector<unsigned long long> nnz(A);
    CU(ctx, cudaMemcpyAsync(nnz.data(), d_nnz.p, A * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    col_ptr[0] = 0;
    for (uint32_t a = 0; a < A; a++) col_ptr[a + 1] = col_ptr[a] + (int64_t)nnz[a];
    const uint64_t n = (uint64_t)col_ptr[A];
    if (!value || n == 0) return GATB_OK;
    if (capacity < n)
        return fail(ctx, GATB_ERR_CAPACITY, "colacc_export: " + std::to_string(n) + " non-zero bins, capacity " +
                                                std::to_string(capacity));
    DevBuf<long long> d_ptr;
    DevBuf<uint32_t> d_value;
    DevBuf<unsigned long long> d_count;
    CU(ctx, d_ptr.upload((const long long *)col_ptr, (size_t)A + 1, st));
    CU(ctx, d_value.alloc(n));
    CU(ctx, d_count.alloc(n));
    p.col_ptr = d_ptr.p; p.value = d_value.p; p.count = d_count.p;
    { ProfScope ps(ctx, PROF_OTHER); CU(ctx, launch_colacc_export(st, p, true)); }
    CU(ctx, cudaMemcpyAsync(value, d_value.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaMemcpyAsync(count, d_count.p, n * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    return GATB_OK;
}

extern "C" int gatb_colacc_add_sparse(gatb_colacc *c, const int64_t *col_ptr, const uint32_t *value, const uint64_t *count)
{
    if (!c || !col_ptr) return GATB_ERR_INVALID;
    gatb_ctx *ctx = c->ctx;
    const uint32_t A = c->A;
    if (col_ptr[0] != 0) return fail(ctx, GATB_ERR_INVALID, "colacc_add_sparse: col_ptr[0] is not 0");
    for (uint32_t a = 0; a < A; a++)
        if (col_ptr[a + 1] < col_ptr[a]) return fail(ctx, GATB_ERR_INVALID, "colacc_add_sparse: col_ptr decreases");
    const uint64_t n = (uint64_t)col_ptr[A];
    if (n == 0) return GATB_OK;
    if (!value || !count) return GATB_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    ColSparseParams p = sparse_params(c);
    DevBuf<long long> d_ptr;
    DevBuf<uint32_t> d_value, d_error;
    DevBuf<unsigned long long> d_count;
    CU(ctx, d_ptr.upload((const long long *)col_ptr, (size_t)A + 1, st));
    CU(ctx, d_value.upload(value, n, st));
    CU(ctx, d_count.upload((const unsigned long long *)count, n, st));
    CU(ctx, d_error.alloc(1));
    CU(ctx, cudaMemsetAsync(d_error.p, 0, sizeof(uint32_t), st));
    p.col_ptr = d_ptr.p; p.value = d_value.p; p.count = d_count.p; p.n_entries = n; p.error = d_error.p;
    uint32_t error = 0;
    { ProfScope ps(ctx, PROF_OTHER); CU(ctx, launch_colacc_add_sparse(st, p, false)); }
    CU(ctx, cudaMemcpyAsync(&error, d_error.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    if (error) return fail(ctx, GATB_ERR_RANGE, "colacc_add_sparse: a histogram value lies outside the window of its "
                                                "column, or a count is 2^32 or more");
    { ProfScope ps(ctx, PROF_OTHER); CU(ctx, launch_colacc_add_sparse(st, p, true)); }
    return GATB_OK;
}

extern "C" int gatb_colacc_finish(gatb_colacc *c, double pseudo_count, double *expected, double *stddev, double *lower95,
                                  double *upper95, double *fold, double *pvalue, uint8_t *missed)
{
    if (!c) return GATB_ERR_INVALID;
    gatb_ctx *ctx = c->ctx;
    const uint32_t A = c->A;
    const uint64_t l = c->l;
    if (c->sums.rows != l)
        return fail(ctx, GATB_ERR_INVALID, "colacc_finish: the sums hold " + std::to_string(c->sums.rows) + " of " +
                                               std::to_string(l) + " samples");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    DevBuf<uint32_t> d_q;                           // q [2][A] | missed [A]
    DevBuf<unsigned long long> d_total;
    CU(ctx, d_q.alloc(3 * (size_t)A));
    CU(ctx, d_total.alloc(A));
    ColHistParams h;
    memset(&h, 0, sizeof(h));
    h.n_cols = A; h.lo = c->win.p; h.width = c->win.p + A; h.bin_off = c->bin_off.p; h.bins = c->bins.p;
    h.outside = c->outside.p;
    h.n_samples = l; ci_ranks(l, h.rank_lo, h.rank_hi);
    h.q = d_q.p; h.missed = d_q.p + 2 * (size_t)A; h.total = d_total.p;
    { ProfScope ps(ctx, PROF_OTHER); CU(ctx, launch_colacc_pick(st, h)); }
    std::vector<unsigned long long> total(A);
    std::vector<uint32_t> q(3 * (size_t)A);
    CU(ctx, cudaMemcpyAsync(q.data(), d_q.p, q.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaMemcpyAsync(total.data(), d_total.p, A * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    std::vector<double> mean, sq, qlo(A), qhi(A);
    if (const int rc = c->sums.read(l, mean, sq)) return rc;       // (synchronises the stream: q and total are here)
    for (uint32_t a = 0; a < A; a++) {
        if (total[a] != l)
            return fail(ctx, GATB_ERR_INVALID, "colacc_finish: the histogram of column " + std::to_string(a) + " holds " +
                                                   std::to_string(total[a]) + " of " + std::to_string(l) + " samples");
        const bool miss = q[2 * (size_t)A + a] != 0;
        qlo[a] = miss ? NAN : (double)q[a];
        qhi[a] = miss ? NAN : (double)q[A + a];
        if (missed) missed[a] = miss ? 1 : 0;
    }
    finish_columns(l, A, c->observed.data(), c->sums.obs_eff.data(), c->ref.empty() ? nullptr : c->ref.data(), pseudo_count,
                   mean.data(), sq.data(), qlo.data(), qhi.data(), c->sums.host(ColumnSums::N_LT),
                   c->sums.host(ColumnSums::N_EQ), expected, stddev, lower95, upper95, fold, pvalue);
    return GATB_OK;
}

extern "C" void gatb_colacc_destroy(gatb_colacc *c)
{
    if (!c) return;
    cudaSetDevice(c->ctx->device);
    tl_stream = c->ctx->stream;
    delete c;                                       // (the buffers go back to the pool in stream order)
}

// ---------------------------------------------------------------------------------------------------
// Westfall-Young step-down minP over one family of columns (DESIGN.md §11): a column accumulator counts the sums and
// extremes, then the histograms over every column's [min, max]; the table pass turns the histograms into K_a(v), the
// host orders the family by its thresholds K_a(v_a), and the rows pass counts C_j.  Integers up to the last division.
extern "C" int gatb_westfall_young(gatb_ctx *ctx, const uint32_t *counts, uint64_t n_samples, uint64_t row_stride,
                                   int n_cols, const double *observed, const double *ref_fold, uint64_t arena_budget,
                                   double *pvalue, double *adjusted)
{
    if (!ctx || !counts || !observed || !adjusted || n_cols <= 0) return GATB_ERR_INVALID;
    if (row_stride < (uint64_t)n_cols) return fail(ctx, GATB_ERR_INVALID, "westfall_young: row_stride < n_cols");
    const uint32_t A = (uint32_t)n_cols;
    const uint64_t l = n_samples;
    gatb_colacc *raw = nullptr;
    if (const int rc = gatb_colacc_create(ctx, n_cols, l, observed, ref_fold, &raw)) return rc;
    std::unique_ptr<gatb_colacc, void (*)(gatb_colacc *)> c(raw, gatb_colacc_destroy);
    cudaStream_t st = ctx->stream;
    if (const int rc = gatb_colacc_add(raw, counts, l, row_stride, GATB_COLACC_SUMS)) return rc;
    std::vector<double> mean, sq;
    if (const int rc = raw->sums.read(l, mean, sq)) return rc;
    // the windows: every column's [min, max]
    std::vector<uint32_t> lo(A), width(A);
    uint64_t arena = 0;
    for (uint32_t a = 0; a < A; a++) {
        const uint64_t w = (uint64_t)raw->sums.h_mm[A + a] - raw->sums.h_mm[a] + 1u;
        arena += 4u * w;
        lo[a] = raw->sums.h_mm[a];
        width[a] = (uint32_t)std::min<uint64_t>(w, 0xffffffffu);
    }
    if (arena > arena_budget)
        return fail(ctx, GATB_ERR_CAPACITY, "westfall_young: the [min, max] windows need " + std::to_string(arena) +
                                                " bytes of histogram bins, more than the " + std::to_string(arena_budget) +
                                                " bytes allowed (" + std::to_string(A) + " columns)");
    for (uint32_t a = 0; a < A; a++)
        if (raw->sums.h_mm[a] == 0u && raw->sums.h_mm[A + a] == 0xffffffffu)
            return fail(ctx, GATB_ERR_CAPACITY, "westfall_young: a column spans all 2^32 values");
    if (const int rc = gatb_colacc_set_windows(raw, lo.data(), width.data())) return rc;
    if (const int rc = gatb_colacc_add(raw, counts, l, row_stride, GATB_COLACC_HIST)) return rc;
    // the thresholds K_a(v_a) against each column's expected value, and the order of the family
    std::vector<double> expected(A);
    std::vector<uint32_t> thr(A);
    const unsigned long long *n_lt = raw->sums.host(ColumnSums::N_LT), *n_eq = raw->sums.host(ColumnSums::N_EQ);
    for (uint32_t a = 0; a < A; a++) {
        expected[a] = ref_fold ? mean[a] * ref_fold[a] : mean[a];
        thr[a] = (uint32_t)std::max<uint64_t>(1, two_sided_index(l, n_lt[a], n_eq[a], raw->sums.obs_eff[a], expected[a]));
        if (pvalue) pvalue[a] = two_sided_pvalue(l, n_lt[a], n_eq[a], raw->sums.obs_eff[a], expected[a]);
    }
    std::vector<uint32_t> order(A);
    for (uint32_t a = 0; a < A; a++) order[a] = a;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return thr[x] < thr[y]; });
    std::vector<uint32_t> pos(2 * (size_t)A);                // col | thr, per position
    std::vector<long long> base(A);
    std::vector<unsigned long long> bin_off(A);
    uint64_t off = 0;
    for (uint32_t a = 0; a < A; a++) { bin_off[a] = off; off += width[a]; }
    for (uint32_t j = 0; j < A; j++) {
        const uint32_t a = order[j];
        pos[j] = a; pos[A + j] = thr[a];
        base[j] = (long long)bin_off[a] - (long long)lo[a];
    }
    DevBuf<double> d_expected;
    DevBuf<uint32_t> d_pos, d_hits;
    DevBuf<long long> d_base;
    CU(ctx, d_expected.upload(expected.data(), A, st));
    CU(ctx, d_pos.upload(pos.data(), pos.size(), st));
    CU(ctx, d_base.upload(base.data(), A, st));
    CU(ctx, d_hits.alloc(A));
    CU(ctx, cudaMemsetAsync(d_hits.p, 0, A * sizeof(uint32_t), st));
    WestfallYoungParams p;
    memset(&p, 0, sizeof(p));
    p.counts = counts; p.n_rows = l; p.row_stride = row_stride; p.n_cols = A;
    p.lo = raw->win.p; p.width = raw->win.p + A; p.bin_off = raw->bin_off.p; p.expected = d_expected.p; p.bins = raw->bins.p;
    p.col = d_pos.p; p.thr = d_pos.p + A; p.base = d_base.p; p.hits = d_hits.p;
    { ProfScope ps(ctx, PROF_OTHER); CU(ctx, launch_westfall_young_table(st, p)); }
    { ProfScope ps(ctx, PROF_OTHER); CU(ctx, launch_westfall_young_rows(st, p, ctx->sm_count)); }
    std::vector<uint32_t> hits(A);
    CU(ctx, cudaMemcpyAsync(hits.data(), d_hits.p, A * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    // the step-down: the running max of max(1, C_i) over the positions up to j, then the one division
    uint32_t run = 1;
    for (uint32_t j = 0; j < A; j++) {
        run = std::max(run, hits[j]);
        adjusted[order[j]] = (double)run / (double)l;
    }
    return GATB_OK;
}

// ---------------------------------------------------------------------------------------------------
// gat-compare: statistics of the sampled log ratio of two fold-change columns, pair by pair.  m1 / m2: device matrices,
// uint32 or float64 each (is_float1 / is_float2); the derived samples are the same doubles either way
static int compare_stats(gatb_ctx *ctx, uint64_t n_samples, const void *m1, int is_float1, int n_cols1, const void *m2,
                         int is_float2, int n_cols2, uint64_t n_pairs, const int32_t *col1, const int32_t *col2,
                         const double *obs1, const double *obs2, const double *delta, double pseudo_count,
                         double *expected, double *stddev, double *lower95, double *upper95, double *fold, double *pvalue)
{
    cudaStream_t st = ctx->stream;
    DevBuf<double> d_o1, d_o2, d_delta, d_out;
    DevBuf<int32_t> d_c1, d_c2;
    CU(ctx, d_c1.upload(col1, n_pairs, st)); CU(ctx, d_c2.upload(col2, n_pairs, st));
    CU(ctx, d_o1.upload(obs1, n_pairs, st)); CU(ctx, d_o2.upload(obs2, n_pairs, st));
    CU(ctx, d_delta.upload(delta, n_pairs, st));
    // pairs in chunks of at most ~256 MB of derived samples
    const uint64_t chunk = std::max<uint64_t>(1, std::min<uint64_t>(n_pairs, (256ull << 20) / (8ull * n_samples)));
    CU(ctx, d_out.alloc(chunk * n_samples));
    for (uint64_t p0 = 0; p0 < n_pairs; p0 += chunk) {
        const uint32_t np = (uint32_t)std::min<uint64_t>(chunk, n_pairs - p0);
        CompareParams cp;
        cp.m1 = m1; cp.m2 = m2; cp.is_float1 = is_float1; cp.is_float2 = is_float2;
        cp.n_cols1 = (uint32_t)n_cols1; cp.n_cols2 = (uint32_t)n_cols2; cp.n_samples = n_samples;
        cp.col1 = d_c1.p + p0; cp.col2 = d_c2.p + p0;
        cp.obs1 = d_o1.p + p0; cp.obs2 = d_o2.p + p0; cp.delta = d_delta.p + p0;
        cp.n_pairs = np; cp.pseudo_count = pseudo_count; cp.out = d_out.p;
        { ProfScope ps(ctx, PROF_OTHER); launch_compare_derive(st, cp); }
        CU(ctx, cudaGetLastError());
        // AnnotatorResult(..., observed_delta_fold, sampled_delta_fold, pseudo_count=0)
        int rc = gatb_column_stats(ctx, d_out.p, 1, 1, n_samples, (int)np, delta + p0, nullptr, 0.0,
                                   expected ? expected + p0 : nullptr, stddev ? stddev + p0 : nullptr,
                                   lower95 ? lower95 + p0 : nullptr, upper95 ? upper95 + p0 : nullptr,
                                   fold ? fold + p0 : nullptr, pvalue ? pvalue + p0 : nullptr);
        if (rc) return rc;
    }
    return GATB_OK;
}

static int compare_check(gatb_ctx *ctx, uint64_t n_samples, int n_cols1, int n_cols2, uint64_t n_pairs, const int32_t *col1,
                         const int32_t *col2)
{
    if (n_samples < 1) return fail(ctx, GATB_ERR_INVALID, "compare_stats: no samples");
    for (uint64_t q = 0; q < n_pairs; q++)
        if (col1[q] < 0 || col1[q] >= n_cols1 || col2[q] < 0 || col2[q] >= n_cols2)
            return fail(ctx, GATB_ERR_INVALID, "compare_stats: column index out of range");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    return GATB_OK;
}

extern "C" int gatb_compare_stats(gatb_ctx *ctx, uint64_t n_samples, const double *m1, int n_cols1,
                                  const double *m2, int n_cols2, uint64_t n_pairs, const int32_t *col1,
                                  const int32_t *col2, const double *obs1, const double *obs2, const double *delta,
                                  double pseudo_count, double *expected, double *stddev, double *lower95,
                                  double *upper95, double *fold, double *pvalue)
{
    if (!ctx || !m1 || !m2 || !col1 || !col2 || !obs1 || !obs2 || !delta || n_cols1 <= 0 || n_cols2 <= 0)
        return GATB_ERR_INVALID;
    if (const int rc = compare_check(ctx, n_samples, n_cols1, n_cols2, n_pairs, col1, col2)) return rc;
    if (n_pairs == 0) return GATB_OK;
    DevBuf<double> d_m1, d_m2;
    CU(ctx, d_m1.upload(m1, n_samples * (uint64_t)n_cols1, ctx->stream));
    if (m2 != m1) CU(ctx, d_m2.upload(m2, n_samples * (uint64_t)n_cols2, ctx->stream));
    return compare_stats(ctx, n_samples, d_m1.p, 1, n_cols1, m2 != m1 ? d_m2.p : d_m1.p, 1, n_cols2, n_pairs, col1, col2,
                         obs1, obs2, delta, pseudo_count, expected, stddev, lower95, upper95, fold, pvalue);
}

extern "C" int gatb_compare_stats_device(gatb_ctx *ctx, uint64_t n_samples, const void *m1, int is_float1, int n_cols1,
                                         const void *m2, int is_float2, int n_cols2, uint64_t n_pairs, const int32_t *col1,
                                         const int32_t *col2, const double *obs1, const double *obs2, const double *delta,
                                         double pseudo_count, double *expected, double *stddev, double *lower95,
                                         double *upper95, double *fold, double *pvalue)
{
    if (!ctx || !m1 || !m2 || !col1 || !col2 || !obs1 || !obs2 || !delta || n_cols1 <= 0 || n_cols2 <= 0)
        return GATB_ERR_INVALID;
    if (const int rc = compare_check(ctx, n_samples, n_cols1, n_cols2, n_pairs, col1, col2)) return rc;
    if (n_pairs == 0) return GATB_OK;
    return compare_stats(ctx, n_samples, m1, is_float1 ? 1 : 0, n_cols1, m2, is_float2 ? 1 : 0, n_cols2, n_pairs, col1, col2,
                         obs1, obs2, delta, pseudo_count, expected, stddev, lower95, upper95, fold, pvalue);
}

// ---------------------------------------------------------------------------------------------------
// counts table text (--output-counts-pattern)
extern "C" int gatb_format_counts(gatb_ctx *ctx, const uint32_t *counts, int counts_is_device, uint64_t n_samples,
                                  int n_cols, uint64_t *col_off, char *text, uint64_t capacity)
{
    if (!ctx || !counts || !col_off || n_cols <= 0) return GATB_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    const uint32_t A = (uint32_t)n_cols;
    DevBuf<uint32_t> d_counts;
    const uint32_t *dc = counts;
    if (!counts_is_device) {
        CU(ctx, d_counts.upload(counts, n_samples * A, st));
        dc = d_counts.p;
    }
    DevBuf<unsigned long long> d_len, d_off;
    CU(ctx, d_len.alloc(A));
    { ProfScope ps(ctx, PROF_OTHER); launch_format_counts(st, dc, n_samples, A, d_len.p, nullptr, nullptr); }
    CU(ctx, cudaGetLastError());
    std::vector<unsigned long long> h_len(A), h_off(A + 1, 0);
    CU(ctx, cudaMemcpyAsync(h_len.data(), d_len.p, A * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    for (uint32_t a = 0; a < A; a++) h_off[a + 1] = h_off[a] + h_len[a];
    for (uint32_t a = 0; a <= A; a++) col_off[a] = h_off[a];
    if (!text) return GATB_OK;
    if (capacity < h_off[A]) return fail(ctx, GATB_ERR_CAPACITY, "format_counts: text buffer too small");
    if (h_off[A] == 0) return GATB_OK;
    DevBuf<char> d_text;
    CU(ctx, d_off.upload(h_off.data(), A + 1, st));
    CU(ctx, d_text.alloc(h_off[A]));
    { ProfScope ps(ctx, PROF_OTHER); launch_format_counts(st, dc, n_samples, A, nullptr, d_off.p, d_text.p); }
    CU(ctx, cudaGetLastError());
    CU(ctx, cudaMemcpyAsync(text, d_text.p, h_off[A], cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    return GATB_OK;
}

// ---------------------------------------------------------------------------------------------------
// interval lists on the device (input preparation, prep.cu)
#include "prep.cuh"

struct gatb_lists {
    gatb_ctx *ctx = nullptr;
    uint32_t n_lists = 0;
    uint64_t n = 0;                      // intervals
    DevBuf<uint64_t> offs;               // [n_lists + 1]
    DevBuf<uint32_t> start, end, list_of;   // [n]
};

static inline int bits_for(uint64_t x) { int b = 0; while (x) { b++; x >>= 1; } return b; }

// device rows (key = list << 32 | start, val = end; unsorted) -> a new gatb_lists: sort, merge, compact.
// The buffers are consumed.  join_adjacent: 0 = SegmentList.normalize, 1 = merge(0)
static int lists_from_device_rows(gatb_ctx *ctx, DevBuf<uint64_t> &key, DevBuf<uint32_t> &val, uint64_t n, uint32_t n_lists,
                                  int join_adjacent, gatb_lists **out)
{
    cudaStream_t st = ctx->stream;
    gatb_lists *L = new gatb_lists();
    L->ctx = ctx; L->n_lists = n_lists;
    DevBuf<uint64_t> key_alt;
    DevBuf<uint32_t> val_alt, head, head_excl;
    DevBuf<uint8_t> temp;
    cudaError_t e = cudaSuccess;
#define TRY(x) do { if (e == cudaSuccess) e = (x); } while (0)
    TRY(L->offs.alloc((size_t)n_lists + 1));
    if (n == 0) {
        TRY(cudaMemsetAsync(L->offs.p, 0, ((size_t)n_lists + 1) * sizeof(uint64_t), st));
        TRY(cudaStreamSynchronize(st));
        if (e != cudaSuccess) { delete L; return fail(ctx, GATB_ERR_CUDA, cudaGetErrorString(e)); }
        *out = L;
        return GATB_OK;
    }
    MergeRows m;
    memset(&m, 0, sizeof(m));
    m.n = n; m.end_bit = 32 + std::max(1, bits_for(n_lists)); m.join_adjacent = join_adjacent;
    m.temp_bytes = sort_temp_bytes(n, m.end_bit);
    TRY(key_alt.alloc(n)); TRY(val_alt.alloc(n)); TRY(head.alloc(n)); TRY(head_excl.alloc(n)); TRY(temp.alloc(m.temp_bytes));
    if (e != cudaSuccess) { delete L; return fail(ctx, GATB_ERR_CUDA, cudaGetErrorString(e)); }
    m.key = key.p; m.key_alt = key_alt.p; m.val = val.p; m.val_alt = val_alt.p; m.head = head.p; m.head_excl = head_excl.p;
    m.temp = temp.p;
    { ProfScope ps(ctx, PROF_OTHER); ctx->launches += 6; e = merge_sorted_rows(st, m); }
    uint32_t tail[2] = {0, 0};          // exclusive head sum and head flag of the last row -> number of merged segments
    TRY(cudaMemcpyAsync(&tail[0], m.head_excl + (n - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    TRY(cudaMemcpyAsync(&tail[1], m.head + (n - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    TRY(cudaStreamSynchronize(st));
    L->n = (uint64_t)tail[0] + tail[1];
    TRY(L->start.alloc(L->n)); TRY(L->end.alloc(L->n)); TRY(L->list_of.alloc(L->n));
    TRY(cudaMemsetAsync(L->end.p, 0, L->n * sizeof(uint32_t), st));
    if (e == cudaSuccess) {
        ProfScope ps(ctx, PROF_OTHER);
        ctx->launches += 1;
        launch_rows_emit(st, m, n_lists, L->offs.p, L->start.p, L->end.p, L->list_of.p);
        e = cudaGetLastError();
    }
    TRY(cudaStreamSynchronize(st));
#undef TRY
    if (e != cudaSuccess) { delete L; return fail(ctx, GATB_ERR_CUDA, cudaGetErrorString(e)); }
    *out = L;
    return GATB_OK;
}

extern "C" int gatb_lists_from_rows(gatb_ctx *ctx, uint64_t n_rows, const uint32_t *list_id, const uint32_t *start,
                                    const uint32_t *end, uint32_t n_lists, int join_adjacent, gatb_lists **out)
{
    if (!ctx || !out || (n_rows && (!list_id || !start || !end))) return GATB_ERR_INVALID;
    *out = nullptr;
    if (n_rows > 0x7fffffffull) return fail(ctx, GATB_ERR_INVALID, "lists: 2^31 or more rows");
    if (n_lists == 0 || n_lists > 0x7ffffffeu) return fail(ctx, GATB_ERR_INVALID, "lists: need between 1 and 2^31 lists");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    DevBuf<uint32_t> d_l, d_s, d_e, d_err;
    DevBuf<uint64_t> key;
    DevBuf<uint32_t> val;
    CU(ctx, d_l.upload(list_id, n_rows, st)); CU(ctx, d_s.upload(start, n_rows, st)); CU(ctx, d_e.upload(end, n_rows, st));
    CU(ctx, d_err.alloc(1));
    CU(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(uint32_t), st));
    CU(ctx, key.alloc(n_rows)); CU(ctx, val.alloc(n_rows));
    { ProfScope ps(ctx, PROF_OTHER); launch_rows_key(st, d_l.p, d_s.p, d_e.p, n_rows, n_lists, key.p, val.p, d_err.p); }
    uint32_t h_err = 0;
    CU(ctx, cudaMemcpyAsync(&h_err, d_err.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    if (h_err & 8u) return fail(ctx, GATB_ERR_INVALID, "lists: list id out of range");
    if (h_err & 1u) return fail(ctx, GATB_ERR_RANGE, "lists: coordinate >= 2^31");
    if (h_err & 2u) return fail(ctx, GATB_ERR_INVALID, "lists: inverted segment (start > end)");
    d_l.release(); d_s.release(); d_e.release();
    return lists_from_device_rows(ctx, key, val, n_rows, n_lists, join_adjacent, out);
}

extern "C" int gatb_lists_from_csr(gatb_ctx *ctx, uint32_t n_lists, const uint64_t *offs, const uint32_t *start,
                                   const uint32_t *end, gatb_lists **out)
{
    if (!ctx || !out || !offs) return GATB_ERR_INVALID;
    *out = nullptr;
    int rc = check_lists(ctx, "lists", n_lists, offs, start, end);
    if (rc) return rc;
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    gatb_lists *L = new gatb_lists();
    L->ctx = ctx; L->n_lists = n_lists; L->n = offs[n_lists];
    cudaError_t e = L->offs.upload(offs, (size_t)n_lists + 1, st);
    if (e == cudaSuccess) e = L->start.upload(start, L->n, st);
    if (e == cudaSuccess) e = L->end.upload(end, L->n, st);
    if (e == cudaSuccess) e = L->list_of.alloc(L->n);
    if (e == cudaSuccess) { ProfScope ps(ctx, PROF_OTHER); launch_csr_list(st, L->offs.p, n_lists, L->n, L->list_of.p); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { delete L; return fail(ctx, GATB_ERR_CUDA, cudaGetErrorString(e)); }
    *out = L;
    return GATB_OK;
}

extern "C" void gatb_lists_destroy(gatb_lists *L)
{
    if (!L) return;
    cudaSetDevice(L->ctx->device);
    delete L;
}

extern "C" int gatb_lists_info(const gatb_lists *L, uint32_t *n_lists, uint64_t *n_intervals)
{
    if (!L) return GATB_ERR_INVALID;
    if (n_lists) *n_lists = L->n_lists;
    if (n_intervals) *n_intervals = L->n;
    return GATB_OK;
}

extern "C" int gatb_lists_download(const gatb_lists *L, uint64_t *offs, uint32_t *start, uint32_t *end)
{
    if (!L) return GATB_ERR_INVALID;
    gatb_ctx *ctx = L->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    if (offs) CU(ctx, cudaMemcpyAsync(offs, L->offs.p, ((size_t)L->n_lists + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (start && L->n) CU(ctx, cudaMemcpyAsync(start, L->start.p, L->n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    if (end && L->n) CU(ctx, cudaMemcpyAsync(end, L->end.p, L->n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    return GATB_OK;
}

extern "C" int gatb_lists_sizes(const gatb_lists *L, uint64_t *count, uint64_t *bases)
{
    if (!L) return GATB_ERR_INVALID;
    gatb_ctx *ctx = L->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    if (count) {
        std::vector<uint64_t> h((size_t)L->n_lists + 1);
        CU(ctx, cudaMemcpyAsync(h.data(), L->offs.p, h.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaStreamSynchronize(st));
        for (uint32_t l = 0; l < L->n_lists; l++) count[l] = h[l + 1] - h[l];
    }
    if (bases) {
        DevBuf<unsigned long long> d;
        CU(ctx, d.alloc(L->n_lists));
        CU(ctx, cudaMemsetAsync(d.p, 0, L->n_lists * sizeof(unsigned long long), st));
        { ProfScope ps(ctx, PROF_OTHER); launch_sizes(st, L->list_of.p, L->start.p, L->end.p, L->n, d.p); }
        CU(ctx, cudaGetLastError());
        CU(ctx, cudaMemcpyAsync(bases, d.p, L->n_lists * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaStreamSynchronize(st));
    }
    return GATB_OK;
}

extern "C" int gatb_lists_restrict(const gatb_lists *in, uint32_t n_keys, uint32_t fanout, const gatb_lists *other,
                                   int truncate, gatb_lists **out)
{
    if (!in || !other || !out) return GATB_ERR_INVALID;
    *out = nullptr;
    gatb_ctx *ctx = in->ctx;
    if (other->ctx != ctx) return fail(ctx, GATB_ERR_INVALID, "restrict: lists belong to different contexts");
    if (n_keys == 0 || fanout == 0 || in->n_lists % n_keys != 0 || (uint64_t)n_keys * fanout != other->n_lists)
        return fail(ctx, GATB_ERR_INVALID, "restrict: need in.n_lists = tracks * n_keys and other.n_lists = n_keys * fanout");
    if ((uint64_t)in->n_lists * fanout > 0x7ffffffeull || in->n * fanout > 0x7fffffffull)
        return fail(ctx, GATB_ERR_INVALID, "restrict: too many lists / intervals");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    gatb_lists *L = new gatb_lists();
    L->ctx = ctx; L->n_lists = in->n_lists * fanout;
    const uint64_t slots = in->n * fanout;
    DevBuf<uint32_t> cnt, cnt_excl;
    DevBuf<uint8_t> temp;
    cudaError_t e = L->offs.alloc((size_t)L->n_lists + 1);
#define TRY(x) do { if (e == cudaSuccess) e = (x); } while (0)
    RestrictParams p;
    memset(&p, 0, sizeof(p));
    p.in_offs = in->offs.p; p.in_start = in->start.p; p.in_end = in->end.p; p.in_list = in->list_of.p; p.n = in->n;
    p.o_offs = other->offs.p; p.o_start = other->start.p; p.o_end = other->end.p;
    p.n_keys = n_keys; p.fanout = fanout; p.truncate = truncate ? 1 : 0;
    uint64_t total = 0;
    if (slots) {
        const size_t tb = exclusive_sum_bytes(slots, false);
        TRY(cnt.alloc(slots)); TRY(cnt_excl.alloc(slots)); TRY(temp.alloc(tb));
        p.cnt = cnt.p; p.cnt_excl = cnt_excl.p;
        if (e == cudaSuccess) { ProfScope ps(ctx, PROF_OTHER); e = launch_restrict(st, p, false); }
        if (e == cudaSuccess) { ctx->launches += 2; e = exclusive_sum_u32(st, temp.p, tb, cnt.p, cnt_excl.p, slots); }
        uint32_t tail[2] = {0, 0};
        TRY(cudaMemcpyAsync(&tail[0], cnt_excl.p + (slots - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        TRY(cudaMemcpyAsync(&tail[1], cnt.p + (slots - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        TRY(cudaStreamSynchronize(st));
        total = (uint64_t)tail[0] + tail[1];
    }
    L->n = total;
    TRY(L->start.alloc(total)); TRY(L->end.alloc(total)); TRY(L->list_of.alloc(total));
    p.out_offs = L->offs.p; p.out_start = L->start.p; p.out_end = L->end.p; p.out_list = L->list_of.p;
    if (e == cudaSuccess && slots) { ProfScope ps(ctx, PROF_OTHER); e = launch_restrict(st, p, true); }
    if (e == cudaSuccess) {
        if (slots) { ProfScope ps(ctx, PROF_OTHER); launch_restrict_offs(st, p, in->n_lists, total); e = cudaGetLastError(); }
        else e = cudaMemsetAsync(L->offs.p, 0, ((size_t)L->n_lists + 1) * sizeof(uint64_t), st);
    }
    TRY(cudaStreamSynchronize(st));
#undef TRY
    if (e != cudaSuccess) { delete L; return fail(ctx, GATB_ERR_CUDA, cudaGetErrorString(e)); }
    *out = L;
    return GATB_OK;
}

extern "C" int gatb_lists_collapse(const gatb_lists *in, uint32_t fanout, gatb_lists **out)
{
    if (!in || !out) return GATB_ERR_INVALID;
    *out = nullptr;
    gatb_ctx *ctx = in->ctx;
    if (fanout == 0 || in->n_lists % fanout != 0) return fail(ctx, GATB_ERR_INVALID, "collapse: n_lists is not a multiple of fanout");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    DevBuf<uint64_t> key;
    DevBuf<uint32_t> val;
    CU(ctx, key.alloc(in->n)); CU(ctx, val.alloc(in->n));
    { ProfScope ps(ctx, PROF_OTHER); launch_collapse_key(st, in->list_of.p, in->start.p, in->end.p, in->n, fanout, key.p, val.p); }
    CU(ctx, cudaGetLastError());
    return lists_from_device_rows(ctx, key, val, in->n, in->n_lists / fanout, 1, out);
}

extern "C" int gatb_lists_select(const gatb_lists *in, uint32_t n_out, const uint32_t *src, gatb_lists **out)
{
    if (!in || !out || (n_out && !src)) return GATB_ERR_INVALID;
    *out = nullptr;
    gatb_ctx *ctx = in->ctx;
    if (n_out == 0) return fail(ctx, GATB_ERR_INVALID, "select: no lists");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    gatb_lists *L = new gatb_lists();
    L->ctx = ctx; L->n_lists = n_out;
    DevBuf<uint32_t> d_src;
    DevBuf<unsigned long long> len;
    DevBuf<uint8_t> temp;
    const size_t tb = exclusive_sum_bytes((uint64_t)n_out + 1, true);
    cudaError_t e = d_src.upload(src, n_out, st);
#define TRY(x) do { if (e == cudaSuccess) e = (x); } while (0)
    TRY(len.alloc((size_t)n_out + 1)); TRY(temp.alloc(tb)); TRY(L->offs.alloc((size_t)n_out + 1));
    if (e == cudaSuccess) { ProfScope ps(ctx, PROF_OTHER); launch_select_count(st, in->offs.p, d_src.p, n_out, in->n_lists, len.p); e = cudaGetLastError(); }
    if (e == cudaSuccess) {
        ctx->launches += 2;
        e = exclusive_sum_u64(st, temp.p, tb, len.p, reinterpret_cast<unsigned long long *>(L->offs.p), (uint64_t)n_out + 1);
    }
    uint64_t total = 0;
    TRY(cudaMemcpyAsync(&total, L->offs.p + n_out, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    TRY(cudaStreamSynchronize(st));
    L->n = total;
    TRY(L->start.alloc(total)); TRY(L->end.alloc(total)); TRY(L->list_of.alloc(total));
    if (e == cudaSuccess && total) {
        ProfScope ps(ctx, PROF_OTHER);
        launch_select_copy(st, in->offs.p, in->start.p, in->end.p, d_src.p, n_out, in->n_lists,
                           reinterpret_cast<const unsigned long long *>(L->offs.p), L->start.p, L->end.p, L->list_of.p);
        e = cudaGetLastError();
    }
    TRY(cudaStreamSynchronize(st));
#undef TRY
    if (e != cudaSuccess) { delete L; return fail(ctx, GATB_ERR_CUDA, cudaGetErrorString(e)); }
    *out = L;
    return GATB_OK;
}

// annotation set straight from device lists: no host round trip of the intervals (SURVEY 8 f1: "CSR built once")
extern "C" int gatb_annotations_create_from_lists(gatb_ctx *ctx, const gatb_lists *L, int n_annot, int n_keys,
                                                  const uint32_t *key_ws_nseg, gatb_annotations **out)
{
    if (!ctx || !L || !out) return GATB_ERR_INVALID;
    *out = nullptr;
    if (L->ctx != ctx) return fail(ctx, GATB_ERR_INVALID, "annotations: the lists belong to another context");
    if (n_annot <= 0 || n_keys <= 0 || (uint64_t)n_annot * n_keys != L->n_lists)
        return fail(ctx, GATB_ERR_INVALID, "annotations: the lists are not n_annot x n_keys");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    // the few host-side facts the index geometry needs: list sizes, the extent of every list, the mean length
    std::vector<uint64_t> offs((size_t)L->n_lists + 1);
    std::vector<uint32_t> last_end(L->n_lists);
    DevBuf<uint32_t> d_last;
    DevBuf<unsigned long long> d_bases;
    CU(ctx, d_last.alloc(L->n_lists));
    { ProfScope ps(ctx, PROF_OTHER); launch_last_end(st, L->offs.p, L->end.p, L->n_lists, d_last.p); }
    CU(ctx, cudaGetLastError());
    CU(ctx, cudaMemcpyAsync(offs.data(), L->offs.p, offs.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaMemcpyAsync(last_end.data(), d_last.p, L->n_lists * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    std::vector<unsigned long long> bases(L->n_lists);
    CU(ctx, d_bases.alloc(L->n_lists));
    CU(ctx, cudaMemsetAsync(d_bases.p, 0, L->n_lists * sizeof(unsigned long long), st));
    { ProfScope ps(ctx, PROF_OTHER); launch_sizes(st, L->list_of.p, L->start.p, L->end.p, L->n, d_bases.p); }
    CU(ctx, cudaGetLastError());
    CU(ctx, cudaMemcpyAsync(bases.data(), d_bases.p, L->n_lists * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    unsigned long long total = 0;
    for (auto b : bases) total += b;
    const uint64_t mean_len = L->n ? std::max<uint64_t>(1, total / L->n) : 1;
    int rc = annotations_create_common(ctx, n_annot, n_keys, offs.data(), nullptr, nullptr, last_end.data(), mean_len,
                                       L->offs.p, L->start.p, L->end.p, key_ws_nseg, out);
    if (rc) return rc;
    rc = annotations_finish(*out);          // (synchronous: the lists may be destroyed as soon as this returns)
    if (rc) {
        tl_stream = ctx->stream;
        delete *out;
        *out = nullptr;
    }
    return rc;
}

// ---------------------------------------------------------------------------------------------------
// multi-GPU exchange without a collective: output routes and peer memory (include/gat_b200.h)
extern "C" int gatb_set_output_routes(gatb_ctx *ctx, int n_routes, const gatb_route *routes)
{
    if (!ctx || n_routes < 0 || (n_routes && !routes)) return GATB_ERR_INVALID;
    if ((uint32_t)n_routes > GATB_MAX_ROUTES) return fail(ctx, GATB_ERR_INVALID, "at most 16 output routes");
    for (int r = 0; r < n_routes; r++)
        if (!routes[r].base || routes[r].col_begin > routes[r].col_end || routes[r].row_stride < routes[r].col_end - routes[r].col_begin)
            return fail(ctx, GATB_ERR_INVALID, "output route: NULL base, inverted column range or rows narrower than the range");
    ctx->routes.assign(routes, routes + n_routes);
    return GATB_OK;
}

extern "C" int gatb_set_route_mode(gatb_ctx *ctx, int by_kernel)
{
    if (!ctx) return GATB_ERR_INVALID;
    ctx->route_copy = by_kernel == 0;
    return GATB_OK;
}

extern "C" int gatb_peer_alloc(gatb_ctx *ctx, uint64_t bytes, void **ptr, unsigned char *handle)
{
    if (!ctx || !ptr || !handle || bytes == 0) return GATB_ERR_INVALID;
    *ptr = nullptr;
    CU(ctx, cudaSetDevice(ctx->device));
    void *p = nullptr;
    CU(ctx, cudaMalloc(&p, bytes));             // (plain cudaMalloc: pool memory cannot be shared through IPC handles)
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return fail(ctx, GATB_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e)); }
    static_assert(sizeof(cudaIpcMemHandle_t) == GATB_PEER_HANDLE_BYTES, "handle size");
    memcpy(handle, &h, sizeof(h));
    *ptr = p;
    return GATB_OK;
}

extern "C" int gatb_peer_free(gatb_ctx *ctx, void *ptr)
{
    if (!ctx) return GATB_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    if (ptr) CU(ctx, cudaFree(ptr));
    return GATB_OK;
}

extern "C" int gatb_peer_open(gatb_ctx *ctx, const unsigned char *handle, void **ptr)
{
    if (!ctx || !handle || !ptr) return GATB_ERR_INVALID;
    *ptr = nullptr;
    CU(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    void *p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(ctx, GATB_ERR_CUDA, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e)); }
    *ptr = p;
    return GATB_OK;
}

extern "C" int gatb_peer_close(gatb_ctx *ctx, void *ptr)
{
    if (!ctx) return GATB_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    if (ptr) CU(ctx, cudaIpcCloseMemHandle(ptr));
    return GATB_OK;
}

// ---------------------------------------------------------------------------------------------------
// counts table reader (--input-counts-file, gat-compare): the passes of count.cu ("counts table parsing").  The first
// call (counts == NULL) checks the grammar; the second repeats the passes and stores the numbers, so that no state
// lives between the calls (the passes cost a few reads of the text).
extern "C" int gatb_parse_counts(gatb_ctx *ctx, const char *text, uint64_t n_bytes, uint64_t line_capacity,
                                 uint64_t *n_rows, uint64_t *n_samples, int *plain, uint64_t *bad_offset,
                                 uint64_t *lines, uint32_t *counts)
{
    if (!ctx || (!text && n_bytes) || !n_rows || !n_samples || !plain || !bad_offset || (line_capacity && !lines))
        return GATB_ERR_INVALID;
    *n_rows = 0; *n_samples = 0; *plain = 1; *bad_offset = PARSE_NONE;
    if (n_bytes == 0) return counts ? fail(ctx, GATB_ERR_INVALID, "parse_counts: empty table") : GATB_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    tl_stream = ctx->stream;
    cudaStream_t st = ctx->stream;
    ParseParams p;
    memset(&p, 0, sizeof(p));
    p.text = (const uint8_t *)text; p.n = n_bytes;
    p.n_tiles = (n_bytes + PARSE_TILE - 1) / PARSE_TILE;
    const uint64_t nt1 = p.n_tiles + 1;
    DevBuf<unsigned long long> d_tiles, d_lines;
    DevBuf<uint8_t> scan_tmp;
    CU(ctx, d_tiles.alloc(3 * nt1 + 1));
    CU(ctx, cudaMemsetAsync(d_tiles.p, 0, 3 * nt1 * sizeof(unsigned long long), st));
    CU(ctx, cudaMemsetAsync(d_tiles.p + 3 * nt1, 0xff, sizeof(unsigned long long), st));
    p.tile_nl = d_tiles.p; p.tile_tab = d_tiles.p + nt1; p.tile_comma = d_tiles.p + 2 * nt1; p.bad = d_tiles.p + 3 * nt1;
    const size_t scan_bytes = parse_scan_bytes(p.n_tiles);
    CU(ctx, scan_tmp.alloc(std::max<size_t>(scan_bytes, 1)));
    { ProfScope ps(ctx, PROF_OTHER); CU(ctx, launch_parse_tiles(st, p, scan_tmp.p, scan_bytes)); }
    unsigned long long bad = PARSE_NONE;
    CU(ctx, cudaMemcpyAsync(&p.n_lines, p.tile_nl + p.n_tiles, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    if (p.n_lines) {
        const uint64_t R = p.n_lines;
        CU(ctx, d_lines.alloc(5 * R));
        p.line_end = d_lines.p; p.tabs_end = d_lines.p + R; p.commas_end = d_lines.p + 2 * R;
        p.counts_start = d_lines.p + 3 * R; p.comma0 = d_lines.p + 4 * R;
        CU(ctx, cudaMemsetAsync(p.counts_start, 0xff, R * sizeof(unsigned long long), st));
        CU(ctx, cudaMemsetAsync(p.comma0, 0, R * sizeof(unsigned long long), st));
        { ProfScope ps(ctx, PROF_OTHER); CU(ctx, launch_parse_marks(st, p)); }
        { ProfScope ps(ctx, PROF_OTHER); CU(ctx, launch_parse_lines(st, p)); }
        unsigned long long first[3];                    // the first line: commas at its end, counts start, commas before it
        CU(ctx, cudaMemcpyAsync(first, p.commas_end, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaMemcpyAsync(first + 1, p.counts_start, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaMemcpyAsync(first + 2, p.comma0, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaMemcpyAsync(&bad, p.bad, sizeof(bad), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaStreamSynchronize(st));
        p.n_values = first[1] == PARSE_NONE ? 0 : first[0] - first[2] + 1;
    } else bad = 0;                                     // no '\n' at all: one unterminated line
    DevBuf<uint32_t> d_rows;                            // [line][value]
    if (p.n_lines && counts && bad == PARSE_NONE) {
        CU(ctx, d_rows.alloc(p.n_lines * p.n_values));
        p.values = d_rows.p;
    }
    if (p.n_lines) {
        { ProfScope ps(ctx, PROF_OTHER); CU(ctx, launch_parse_values(st, p)); }
        CU(ctx, cudaMemcpyAsync(&bad, p.bad, sizeof(bad), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaStreamSynchronize(st));
    }
    *plain = bad == PARSE_NONE;
    *bad_offset = bad;
    if (!*plain) return counts ? fail(ctx, GATB_ERR_INVALID, "parse_counts: not a plain counts table (offending byte at offset " +
                                                                 std::to_string(bad) + ")") : GATB_OK;
    *n_rows = p.n_lines; *n_samples = p.n_values;
    if (lines) {
        const uint64_t R = std::min<uint64_t>(p.n_lines, line_capacity);
        std::vector<unsigned long long> h(2 * R);
        CU(ctx, cudaMemcpyAsync(h.data(), p.line_end, R * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaMemcpyAsync(h.data() + R, p.counts_start, R * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaStreamSynchronize(st));
        for (uint64_t l = 0; l < R; l++) { lines[2 * l] = l ? h[l - 1] + 1 : 0; lines[2 * l + 1] = h[R + l]; }
    }
    if (counts) {
        { ProfScope ps(ctx, PROF_OTHER); CU(ctx, launch_transpose_u32(st, p.values, p.n_lines, p.n_values, counts)); }
        CU(ctx, cudaStreamSynchronize(st));
    }
    if (p.n_lines > line_capacity) return fail(ctx, GATB_ERR_CAPACITY, "parse_counts: line table too small");
    return GATB_OK;
}
