// rtb_abi.cu -- implementation of the C ABI declared in include/rtb.h (librtb200.so).
// Host glue only: argument validation, upload of the flattened scene, kernel launches on the
// context stream, CUDA-event timing, and the host<->device copies of the host-buffer calls.
// There is no CPU path in this library.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <chrono>
#include <vector>

#include "rtb_launch.h"
#include "rtb_misc.cuh"
#include "rtb_build_grid.cuh"
#include "rtb_build_kd.cuh"
#include "rtb_build_bvh.cuh"

#ifndef RTB_SPLIT_MAX_TILES
#define RTB_SPLIT_MAX_TILES 200000 // shards up to 6.4 Mpixel (half a 4K frame) count as "small": their latency-critical tiles go
                                   // to the 8 / 16-lane tier (k-d) or to 4 warps of 8 lanes (grids).  1/2 shard of the 4K SAH frame, kernel
                                   // ms: resumable tier 3.07, no tier 3.51, 8-lane tier 2.80 (profiles/r02_sweep_tiers.log)
#endif
#ifndef RTB_HEAVY_BUCKETS_SMALL
#define RTB_HEAVY_BUCKETS_SMALL 4   // quarter-octaves below the heaviest tile: 4 / 6 / 10 -> slowest 1/8 SAH shard 1.18 / 1.24 / 1.24 ms
#endif
#ifndef RTB_HEAVY_ALPHA
#define RTB_HEAVY_ALPHA 0.0f
#endif
#ifndef RTB_HEAVY_FRACTION_SMALL
#define RTB_HEAVY_FRACTION_SMALL 128 //    quarter-octaves and 1/32 .. 1/8 of the shard measured slower)
#endif
static int splitMaxTiles()
{
    static const int v = getenv("RTB_SPLIT_MAX_TILES") ? atoi(getenv("RTB_SPLIT_MAX_TILES")) : RTB_SPLIT_MAX_TILES;
    return v;
}
// Warp-per-pixel tier (rtb_chain_wide.cuh): how many of the heaviest tiles it takes (wideCount below).
static double tunable(const char *name, double dflt)
{
    const char *v = getenv(name);
    return v ? atof(v) : dflt;
}
// A warp-per-pixel tile costs 2x (regular grid: long cell lists, the lanes are busy) to 4x (k-d trees: 32 lanes
// repeat the node walk) the SM time of the same tile in the throughput kernels and finishes 8-16x sooner, so it
// pays exactly where a frame is bound by the latency of its heaviest chains and not by throughput
// (measured, gpurun_out/sweep2.log, one B200, preset 5, kernel ms without -> with the tier):
//   small frames (400x300):           SAH 1.42 -> 0.49, k-d median 3.55 -> 1.22, regular grid 8.48 -> 0.83
//   regular grid, 1/8 shard of 4K:    worst shard 10.8 -> 4.3;   whole 4K frame 15.6 -> 14.4
//                                     (preset 5's 400x5x400 grid: 33 triangles per occupied cell, `long_lists`; preset 4's
//                                     350x166x400 grid has 4 per cell and 265 cells per ray -- it behaves like the k-d rows)
//   k-d trees, 4K frame or its shards: no gain (the cost distribution is flat: ~1 % of the tiles are within 2x
//                                      of the heaviest, far too many to render this way) -> tier off.
#define RTB_SMALL_FRAME_TILES 16384 // up to 0.5 Mpixel
static int wideCountRaw(int n_tiles, bool long_lists);
// (tier sizes are multiples of four tiles: in group mode, FrameParams::group4, the order is made of groups of four tiles)
static int wideCount(int n_tiles, bool long_lists) { return wideCountRaw(n_tiles, long_lists) & ~3; }
static int wideCountRaw(int n_tiles, bool long_lists)
{
    static const int cap = (int)tunable("RTB_WIDE_CAP", -1), fraction = (int)tunable("RTB_WIDE_FRACTION", 32); // tuning overrides
    if (cap >= 0) return n_tiles / (fraction < 1 ? 1 : fraction) < cap ? n_tiles / (fraction < 1 ? 1 : fraction) : cap;
    if (n_tiles <= RTB_SMALL_FRAME_TILES) return n_tiles / (long_lists ? 16 : 32);
    // shards of a big frame: two tiles per SM.  (Round 1 took up to 1,184 here, tuned on row shards; with column-block
    // shards every rank holds 1 / N of the vanishing-point tiles and the tier's own instructions -- ~4.7 M per tile --
    // become the shard's critical path: slowest 1/8 shard of the 4K frame, kernel ms at 148 / 296 / 592 / 1,184 / 2,368
    // tiles: 3.20 / 2.70 / 2.79 / 3.50 / 4.66, profiles/r02_sweep_tiers.log)
    if (long_lists) return n_tiles <= RTB_SPLIT_MAX_TILES ? (n_tiles / 32 < 296 ? n_tiles / 32 : 296) : 148;
    return 0;
}
// ... of a small shard: how far below the heaviest tile the latency-critical set reaches.  SAH trees: 4 quarter-octaves (2x);
// k-d median trees have a flatter cost distribution and want 6 (2.8x) -- slowest 1/8 shard of the 4K frame with 4 / 6:
// SAH 1.18 / 1.24 ms, median 3.24 / 2.14 ms (profiles/r02_sweep_tiers.log)
static int heavyBucketsSmall(int accel)
{
    static const int forced = (int)tunable("RTB_HEAVY_BUCKETS_SMALL", -1);
    if (forced >= 0) return forced;
    return accel == RTB_ACCEL_KD_MEDIAN ? 6 : RTB_HEAVY_BUCKETS_SMALL;
}
static int heavyFractionSmall() { static const int v = (int)tunable("RTB_HEAVY_FRACTION_SMALL", RTB_HEAVY_FRACTION_SMALL); return v < 1 ? 1 : v; }
// > 0: the latency-critical set of a small shard is chosen by time (k_cost_offsets: tiles whose recorded cost exceeds alpha x the
// balanced finishing time of the kernel); 0: by distance from the heaviest tile (heavyBucketsSmall)
static float heavyAlpha() { static const float v = (float)tunable("RTB_HEAVY_ALPHA", RTB_HEAVY_ALPHA); return v; }
// Size limit of the resumable-walk tier.  Small frames have none: there the warp-per-pixel tier takes the heavy
// tiles and a third kernel in between measured slower (k-d median 400x300: 1.4 ms without, 2.2 ms with).
static int heavyLimitRaw(int n_tiles);
static int heavyLimit(int n_tiles) { return heavyLimitRaw(n_tiles) & ~3; }
static int heavyLimitRaw(int n_tiles)
{
    static const int forced = (int)tunable("RTB_HEAVY_LIMIT", -1);
    if (forced >= 0) return forced;
    if (n_tiles <= RTB_SMALL_FRAME_TILES) return 0;
    // A whole 4K frame is throughput-bound: heaviest-first order alone is best there, any tier costs more warp-instructions than
    // its shorter tail saves (4K frame, kernel ms with / without the resumable tier: SAH 5.03 / 4.70, k-d median 12.45 / 12.18,
    // flat grid 19.5 / 18.8)
    if (n_tiles > splitMaxTiles()) return 0;
    return n_tiles / heavyFractionSmall();
}

using namespace rtb;

struct OrderKey
{
    long long v[10];
    unsigned long long scene_signature; // content signature (rtb_scene_upload): a re-upload of the same scene keeps the order
    rtb_camera cam;
};

// A few worker threads that sleep on a condition variable between jobs.  Two users: an rtb_multi (one worker per device beyond
// the first: the per-device halves of an upload or of a frame launch run side by side, the calling thread takes device 0) and
// every context's scene validation (the whole-stream checks of rtb_scene_upload, cut into tasks).  Thread creation costs
// 30-60 us a piece, as much as the work of one task, hence a pool.
struct WorkerPool
{
    std::vector<std::thread> threads;
    std::mutex m;
    std::condition_variable cv_job, cv_done;
    std::function<void(int)> job;
    unsigned long long generation = 0;
    int pending = 0;
    bool stop = false;

    void start(int n_workers)
    {
        for (int w = 1; w <= n_workers; w++)
            threads.emplace_back([this, w]() {
                unsigned long long seen = 0;
                std::unique_lock<std::mutex> lock(m);
                for (;;)
                {
                    cv_job.wait(lock, [&]() { return stop || generation != seen; });
                    if (stop) return;
                    seen = generation;
                    lock.unlock();
                    job(w); // `job` stays untouched until finish() has seen pending == 0
                    lock.lock();
                    if (--pending == 0) cv_done.notify_all();
                }
            });
    }
    int workers() const { return (int)threads.size(); }
    // fn(w) on every worker w = 1 .. workers(); returns at once.  One job at a time: finish() before the next begin().
    void begin(std::function<void(int)> fn)
    {
        if (threads.empty()) return;
        {
            std::lock_guard<std::mutex> lock(m);
            job = std::move(fn);
            pending = (int)threads.size();
            generation++;
        }
        cv_job.notify_all();
    }
    void finish()
    {
        if (threads.empty()) return;
        std::unique_lock<std::mutex> lock(m);
        cv_done.wait(lock, [&]() { return pending == 0; });
    }
    // fn(i) for i = 1 .. workers() on the worker threads, fn(0) on the calling thread; returns when all have returned
    void run(const std::function<void(int)> &fn)
    {
        begin(fn);
        fn(0);
        finish();
    }
    void shutdown()
    {
        {
            std::lock_guard<std::mutex> lock(m);
            stop = true;
        }
        cv_job.notify_all();
        for (std::thread &t : threads) t.join();
        threads.clear();
    }
    ~WorkerPool() { shutdown(); }
};

// rtb_multi_scene_upload: ONE flat scene goes to every device of the set.  The first device's upload (the producer) stages
// each stream once into its page-locked ring (portable: every device copies from it) and publishes the staged address; the
// other devices' uploads (replicas, on worker threads, a step behind the producer) issue their H2D copies from the same
// staged bytes instead of staging 4.5 MB again per device.  The producer also publishes the verdict of the whole-stream
// index checks, which a replica awaits before it launches anything that indexes with those streams.
struct StageShare
{
    static const int kSlots = 64;
    char *slot[kSlots] = {};
    std::atomic<int> produced{0};
    std::atomic<int> verdict{0};   // 0 pending, 1 streams validated, -1 the producer failed
    bool waitSlot(int i) const
    {
        while (produced.load(std::memory_order_acquire) <= i)
        {
            if (verdict.load(std::memory_order_acquire) < 0) return false;
            std::this_thread::yield();
        }
        return true;
    }
    bool waitVerdict() const
    {
        int v;
        while ((v = verdict.load(std::memory_order_acquire)) == 0) std::this_thread::yield();
        return v > 0;
    }
};

struct rtb_ctx
{
    int device = -1;
    cudaStream_t stream = nullptr;
    Counters *d_counters = nullptr;
    rtb_progress_fn progress = nullptr; // rtb_set_progress
    void *progress_user = nullptr;
    cudaStream_t poll = nullptr;        // side stream of the progress reads
    unsigned long long *h_tiles = nullptr;
    Counters *h_counters = nullptr; // page-locked: the read-back of a timed frame must not block the launching thread
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaStream_t aux = nullptr;                 // high-priority side stream of the latency-critical tiles
    cudaEvent_t fork = nullptr, join = nullptr;
    cudaEvent_t last_frame = nullptr;      // recorded behind the last kernel of every frame (waitLastFrame)
    cudaEvent_t caller_ready = nullptr;    // rtb_scene_mesh_update: the caller's stream, awaited by ctx->stream
    cudaStream_t last_frame_stream = nullptr;
    bool frame_pending = false;
    float *d_frame = nullptr; // grow-only device framebuffer of the host-buffer render call
    size_t d_frame_bytes = 0;
    // heaviest-first tile scheduling (rtb_kernels.cuh): cost of the last frame and the order derived from it
    unsigned int *d_cost = nullptr, *d_order = nullptr, *d_hist = nullptr, *d_cursor = nullptr, *d_heavy = nullptr;
    size_t tile_capacity = 0;
    bool order_valid = false;
    bool tiers_ok = true; // false: this frame uses the order but not the latency tiers (camera moved)
    OrderKey order_key = {};
    // page-locked staging ring of rtb_scene_upload: streams are packed / copied into it and leave with truly
    // asynchronous H2D copies (a pageable source makes every cudaMemcpyAsync a staged, partly synchronous copy)
    char *stage = nullptr;
    size_t stage_cap = 0, stage_used = 0;
    WorkerPool *checkers = nullptr;       // threads of the scene validation (started by the first validating upload)
    std::vector<rtb_ctx *> stage_readers; // contexts of the same rtb_multi whose streams copy out of this ring too
    StageShare *share = nullptr; // set for the duration of an rtb_multi_scene_upload
    bool share_producer = false;
    int share_next = 0;          // replica: the next staged stream to take
    bool sources_page_locked = false; // this upload's flat scene allows copies straight out of page-locked arrays
    std::string error;
};

struct rtb_scene
{
    DScene d;
    std::vector<void *> allocs;
    int64_t bytes = 0;     // device bytes held by the scene
    int64_t h2d_bytes = 0; // bytes the upload copied from host memory (the rest is produced on the device)
    bool has_refractive = false;
    bool has_tunnel = false;
    bool has_mesh = false;   // RTB_PRIM_MESH records: the MESH kernel instantiations, no tunnel tiers
    std::vector<int> mesh_prims; // prims indices of the MESH records (rtb_scene_mesh_download)
    // first-order moments of every mesh node slot (rtb_scene_mesh_moments, 4 float4 per slot, parallel to DScene::mesh_nodes):
    // null until that call; kept out of DScene so that no other kernel's parameters change
    const float4 *mesh_moments = nullptr;
    cudaEvent_t last_use = nullptr; // recorded after every launch that reads the scene
    cudaEvent_t ready = nullptr;    // recorded on ctx->stream behind the upload copies
    // rtb_query_rays on the caller's stream: queries are chained among themselves (a query on another stream than the last one
    // waits for it), so `query_use`, recorded behind every query kernel, covers them all.  Not last_use: a query recording it
    // would hide a render still running on another stream, and renders do not wait for queries.
    mutable cudaEvent_t query_use = nullptr;
    mutable cudaStream_t query_stream = nullptr;
    mutable bool queried = false;
    bool direct_sources = false;    // some copies read the caller's page-locked arrays: rtb_scene_free waits for `ready`
    int64_t grid_cells_used = 0, grid_refs = 0, grid_words = 0;
    int64_t kd_nodes = 0, kd_refs = 0; // k-d tree resident on the device (uploaded or built there)
    const uint2 *kd_nodes_plain = nullptr;  // ... in the caller's / the builder's layout (rtb_scene_kd_download); DScene::kd_nodes /
    const uint32_t *kd_tris_plain = nullptr; //     kd_tris are the copy with every leaf list on an even position (padKdLists)
    int kd_levels = 0;
    bool long_lists = false; // regular grid with >= 16 triangle references per occupied cell (tier policy, wideCount)
    unsigned long long signature = 0; // sampled content hash, identifies "the same scene again" for the tile-order cache
};

// FNV-1a over the small records and a strided sample of the big streams: microseconds, and a collision costs
// nothing but a stale tile order (scheduling only)
static unsigned long long fnv(unsigned long long h, const void *p, size_t bytes)
{
    const unsigned char *b = (const unsigned char *)p;
    for (size_t i = 0; i < bytes; i++) h = (h ^ b[i]) * 0x100000001b3ull;
    return h;
}
template <class T> static unsigned long long fnvSampled(unsigned long long h, const T *p, size_t n)
{
    if (!p || n == 0) return fnv(h, &n, sizeof(n));
    const size_t step = n / 509 + 1;
    for (size_t i = 0; i < n; i += step) h = fnv(h, p + i, sizeof(T));
    h = fnv(h, p + (n - 1), sizeof(T));
    return fnv(h, &n, sizeof(n));
}
static unsigned long long sceneSignature(const rtb_flat_scene *f)
{
    unsigned long long h = 0xcbf29ce484222325ull;
    h = fnv(h, f->prims, sizeof(rtb_prim) * (size_t)f->n_prims);
    h = fnv(h, f->materials, sizeof(rtb_material) * (size_t)f->n_materials);
    h = fnv(h, &f->accel, sizeof(f->accel));
    h = fnv(h, &f->grid_build_resolution, sizeof(f->grid_build_resolution));
    h = fnv(h, &f->grid_build_exact, sizeof(f->grid_build_exact));
    h = fnv(h, &f->kd_build_max_depth, sizeof(f->kd_build_max_depth));
    h = fnv(h, &f->kd_build_leaf_size, sizeof(f->kd_build_leaf_size));
    h = fnvSampled(h, f->loose_tri, f->loose_tri ? (size_t)f->n_loose * 12 : 0);
    h = fnvSampled(h, f->tri, f->tri ? (size_t)f->n_tris * 12 : 0);
    if (f->accel == RTB_ACCEL_REGULAR_GRID || f->accel == RTB_ACCEL_FLAT_GRID)
    {
        h = fnv(h, f->grid_origin, sizeof(f->grid_origin)); h = fnv(h, f->grid_cell, sizeof(f->grid_cell)); h = fnv(h, f->grid_dims, sizeof(f->grid_dims));
        h = fnvSampled(h, f->grid_cell_tris, (size_t)f->n_cell_refs);
    }
    else if (f->accel == RTB_ACCEL_KD_MEDIAN || f->accel == RTB_ACCEL_KD_SAH)
    {
        h = fnvSampled(h, f->kd_nodes, f->kd_nodes ? (size_t)f->n_kd_nodes : 0);
        h = fnvSampled(h, f->kd_leaf_tris, f->kd_leaf_tris ? (size_t)f->n_kd_refs : 0);
    }
    return h;
}

static std::string g_error;
static std::mutex g_error_mutex;

static int fail(rtb_ctx *ctx, int code, const std::string &msg)
{
    {
        std::lock_guard<std::mutex> lock(g_error_mutex);
        g_error = msg;
    }
    if (ctx) ctx->error = msg;
    return code;
}

#define CUDA_TRY(ctx, call)                                                                         \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return fail(ctx, RTB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));     \
    } while (0)

extern "C" int rtb_abi_version(void) { return RTB_ABI_VERSION; }

extern "C" const char *rtb_last_error(const rtb_ctx *ctx)
{
    if (ctx) return ctx->error.c_str();
    std::lock_guard<std::mutex> lock(g_error_mutex);
    static thread_local std::string copy;
    copy = g_error;
    return copy.c_str();
}

extern "C" int rtb_init(int device, rtb_ctx **out)
{
    if (!out) return fail(nullptr, RTB_ERR_INVALID, "rtb_init: null output pointer");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, RTB_ERR_NO_DEVICE, std::string("rtb_init: no CUDA device (") + cudaGetErrorString(e) +
                                                    "); this library has no CPU path");
    if (device < 0 || device >= count) return fail(nullptr, RTB_ERR_INVALID, "rtb_init: device index out of range");
    cudaDeviceProp prop;
    CUDA_TRY(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(nullptr, RTB_ERR_NO_DEVICE, "rtb_init: kernels are built for sm_100a only (device is sm_" +
                                                    std::to_string(prop.major * 10 + prop.minor) + ")");
    rtb_ctx *ctx = new rtb_ctx();
    ctx->device = device;
    CUDA_TRY(ctx, cudaSetDevice(device));
    CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    { // scene buffers come from the stream-ordered pool and are kept for reuse: cudaMalloc/cudaFree cost
      // milliseconds and synchronise the device, which would dominate a per-frame upload
        cudaMemPool_t pool;
        CUDA_TRY(ctx, cudaDeviceGetDefaultMemPool(&pool, device));
        unsigned long long keep = ~0ull;
        CUDA_TRY(ctx, cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    }
    {
        int lo = 0, hi = 0;
        CUDA_TRY(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CUDA_TRY(ctx, cudaStreamCreateWithPriority(&ctx->aux, cudaStreamNonBlocking, hi));
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->fork, cudaEventDisableTiming));
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->join, cudaEventDisableTiming));
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->last_frame, cudaEventDisableTiming));
    }
    CUDA_TRY(ctx, cudaMalloc(&ctx->d_counters, sizeof(Counters)));
    CUDA_TRY(ctx, cudaHostAlloc((void **)&ctx->h_counters, sizeof(Counters), cudaHostAllocDefault));
    for (int i = 0; i < 4; i++) CUDA_TRY(ctx, cudaEventCreate(&ctx->ev[i]));
    *out = ctx;
    return RTB_OK;
}

extern "C" int rtb_shutdown(rtb_ctx *ctx)
{
    if (!ctx) return RTB_OK;
    cudaSetDevice(ctx->device);
    if (ctx->frame_pending) cudaEventSynchronize(ctx->last_frame); // a frame on a caller's stream
    cudaStreamSynchronize(ctx->stream);
    if (ctx->last_frame) cudaEventDestroy(ctx->last_frame);
    if (ctx->caller_ready) cudaEventDestroy(ctx->caller_ready);
    for (int i = 0; i < 4; i++)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->aux) { cudaStreamSynchronize(ctx->aux); cudaStreamDestroy(ctx->aux); }
    if (ctx->fork) cudaEventDestroy(ctx->fork);
    if (ctx->join) cudaEventDestroy(ctx->join);
    if (ctx->d_counters) cudaFree(ctx->d_counters);
    if (ctx->h_counters) cudaFreeHost(ctx->h_counters);
    if (ctx->h_tiles) cudaFreeHost(ctx->h_tiles);
    if (ctx->poll) cudaStreamDestroy(ctx->poll);
    if (ctx->d_frame) cudaFree(ctx->d_frame);
    if (ctx->d_cost) cudaFreeAsync(ctx->d_cost, ctx->stream);
    if (ctx->d_order) cudaFreeAsync(ctx->d_order, ctx->stream);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->d_hist) cudaFree(ctx->d_hist);
    if (ctx->d_cursor) cudaFree(ctx->d_cursor);
    if (ctx->d_heavy) cudaFree(ctx->d_heavy);
    if (ctx->stage) cudaFreeHost(ctx->stage);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx->checkers;
    delete ctx;
    return RTB_OK;
}

static int normRowBlock(const rtb_frame *f) { return f->row_block > 0 ? f->row_block : 8; }

// column-block sharding in effect?  (world > 1 and a column block given)
static bool colSharded(const rtb_frame *f) { return f->col_block > 0 && f->world > 1; }
static bool colShardOk(const rtb_frame *f)
{
    return f->col_block % 8 == 0 && f->width % ((int64_t)f->world * f->col_block) == 0 && !(f->layout & RTB_LAYOUT_REFERENCE);
}

extern "C" int64_t rtb_shard_rows(const rtb_frame *f)
{
    if (!f || f->width <= 0 || f->height <= 0) return -1;
    const int world = f->world > 0 ? f->world : 1, rank = f->rank, rb = normRowBlock(f);
    if (rank < 0 || rank >= world || rb % 8 != 0) return -1;
    if (colSharded(f)) return colShardOk(f) ? f->height : -1; // every rank renders every row
    int64_t rows = 0;
    for (int64_t b = rank; b * rb < f->height; b += world)
    {
        const int64_t y0 = b * rb, y1 = y0 + rb < f->height ? y0 + rb : f->height;
        rows += y1 - y0;
    }
    return rows;
}

extern "C" int64_t rtb_shard_width(const rtb_frame *f)
{
    if (rtb_shard_rows(f) < 0) return -1;
    return colSharded(f) ? f->width / f->world : f->width;
}

// ---- scene upload -----------------------------------------------------------------------------
// `bytes` of page-locked staging memory.  Copies queued from the ring read it asynchronously, so it is only reused
// after the stream has drained (once every few uploads; the ring holds several scenes).
static int stageReserve(rtb_ctx *ctx, size_t bytes, char **out)
{
    bytes = (bytes + 255) & ~(size_t)255;
    if (ctx->stage_used + bytes > ctx->stage_cap)
    {
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        for (rtb_ctx *r : ctx->stage_readers)
        {
            CUDA_TRY(ctx, cudaSetDevice(r->device));
            CUDA_TRY(ctx, cudaStreamSynchronize(r->stream));
        }
        if (!ctx->stage_readers.empty()) CUDA_TRY(ctx, cudaSetDevice(ctx->device));
        if (bytes > ctx->stage_cap)
        {
            if (ctx->stage) cudaFreeHost(ctx->stage);
            ctx->stage = nullptr; ctx->stage_cap = 0;
            const size_t cap = bytes * 2 > ((size_t)64 << 20) ? bytes * 2 : ((size_t)64 << 20);
            CUDA_TRY(ctx, cudaHostAlloc((void **)&ctx->stage, cap, cudaHostAllocPortable)); // every device of an rtb_multi copies from it
            ctx->stage_cap = cap;
        }
        ctx->stage_used = 0;
    }
    *out = ctx->stage + ctx->stage_used;
    ctx->stage_used += bytes;
    return RTB_OK;
}

// is `p` page-locked host memory (cudaHostAlloc / cudaHostRegister)?
static bool pageLocked(const void *p)
{
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) == cudaSuccess && attr.type == cudaMemoryTypeHost) return true;
    cudaGetLastError();
    return false;
}

// `bytes` of staged data: written by fill(char *staging) into this context's ring -- or, for a replica of an
// rtb_multi_scene_upload, the bytes the producer has staged for the same stream (StageShare).
// `src` != nullptr: the staged bytes are a verbatim copy of that caller array -- if the flat scene declares its arrays
// page-locked and stable (rtb_flat_scene.arrays_page_locked) and this one is, the copy reads the array itself (*direct)
template <class Fill>
static int stageFill(rtb_ctx *ctx, size_t bytes, char **out, Fill fill, const void *src = nullptr, bool *direct = nullptr)
{
    StageShare *sh = ctx->share;
    if (sh && !ctx->share_producer)
    {
        const int i = ctx->share_next++;
        if (i >= StageShare::kSlots || !sh->waitSlot(i)) return fail(ctx, RTB_ERR_INVALID, "rtb_multi_scene_upload: the first device's upload failed");
        *out = sh->slot[i];
        if (direct && *out == (const char *)src) *direct = true;
        return RTB_OK;
    }
    if (src && ctx->sources_page_locked && pageLocked(src))
    {
        *out = (char *)const_cast<void *>(src);
        if (direct) *direct = true;
    }
    else
    {
        const int rc = stageReserve(ctx, bytes, out);
        if (rc != RTB_OK) return rc;
        fill(*out);
    }
    if (sh)
    {
        const int i = sh->produced.load(std::memory_order_relaxed);
        if (i >= StageShare::kSlots) return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_multi_scene_upload: too many streams");
        sh->slot[i] = *out;
        sh->produced.store(i + 1, std::memory_order_release);
    }
    return RTB_OK;
}

// device array of n elements; `fill(T *staging)` writes the elements into staging memory (nullptr: zero-filled)
template <class T, class Fill>
static int uploadWith(rtb_ctx *ctx, rtb_scene *s, size_t n, const T **dev, Fill fill, bool zero = false, const T *verbatim = nullptr)
{
    *dev = nullptr;
    const size_t count = n ? n : 1; // keep pointers valid
    void *p = nullptr;
    CUDA_TRY(ctx, cudaMallocAsync(&p, count * sizeof(T), ctx->stream));
    s->allocs.push_back(p);
    s->bytes += (int64_t)(count * sizeof(T));
    if (n && !zero)
    {
        char *st = nullptr;
        const int rc = stageFill(ctx, n * sizeof(T), &st, [&](char *dst) { fill(reinterpret_cast<T *>(dst)); }, verbatim, &s->direct_sources);
        if (rc != RTB_OK) return rc;
        CUDA_TRY(ctx, cudaMemcpyAsync(p, st, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
        s->h2d_bytes += (int64_t)(n * sizeof(T));
    }
    else CUDA_TRY(ctx, cudaMemsetAsync(p, 0, count * sizeof(T), ctx->stream));
    *dev = (const T *)p;
    return RTB_OK;
}

template <class T>
static int uploadArray(rtb_ctx *ctx, rtb_scene *s, const T *host, size_t n, const T **dev)
{
    return uploadWith<T>(ctx, s, n, dev, [&](T *st) { memcpy(st, host, n * sizeof(T)); }, host == nullptr, host);
}

// Triangle records (a, b, c, normal: 12 floats) -> the two device streams, one thread per triangle:
//   exact stream  {a.xyz, e1.x} {e1.yz, e2.xy} {e2.z, n.xyz}; e1 = a - b, e2 = a - c are the float subtractions
//                 reference Triangle.cpp:73-79 performs per test, done once here;
//   pre stream    {a.xyz, A1 eps} {e1.xyz, E eps} {e2.xyz, 0} of the conservative rejection test (rtb_pretest.h).
// Packing 45,900 triangles took 0.7 ms of every upload on the host; here it is one 48-byte read and two 48-byte
// writes per thread behind the raw H2D copy.
__global__ void k_pack_triangles(const float *__restrict__ raw, int n, float4 *__restrict__ exact, float4 *__restrict__ pre)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float t[12];
    const float4 *src = reinterpret_cast<const float4 *>(raw) + 3 * (size_t)i;
    const float4 r0 = src[0], r1 = src[1], r2 = src[2];
    t[0] = r0.x; t[1] = r0.y; t[2] = r0.z; t[3] = r0.w; t[4] = r1.x; t[5] = r1.y; t[6] = r1.z; t[7] = r1.w;
    t[8] = r2.x; t[9] = r2.y; t[10] = r2.z; t[11] = r2.w;
    const float e1x = t[0] - t[3], e1y = t[1] - t[4], e1z = t[2] - t[5];
    const float e2x = t[0] - t[6], e2y = t[1] - t[7], e2z = t[2] - t[8];
    exact[3 * (size_t)i + 0] = make_float4(t[0], t[1], t[2], e1x);
    exact[3 * (size_t)i + 1] = make_float4(e1y, e1z, e2x, e2y);
    exact[3 * (size_t)i + 2] = make_float4(e2z, t[9], t[10], t[11]);
    if (pre)
    {
        const rtb_pre::PreTri p = rtb_pre::makePreTri(t);
        pre[3 * (size_t)i + 0] = make_float4(p.ax, p.ay, p.az, p.a1e);
        pre[3 * (size_t)i + 1] = make_float4(p.e1x, p.e1y, p.e1z, p.ee);
        pre[3 * (size_t)i + 2] = make_float4(p.e2x, p.e2y, p.e2z, 0.f);
    }
}

// raw records -> staging -> device (asynchronous), packed there; `pre` may be null (loose triangles: exact stream only)
// keepRaw != nullptr: the raw device records are handed to the caller (a device accelerator build reads them), who frees them
static int uploadTriangles(rtb_ctx *ctx, rtb_scene *s, const float *host, size_t n, const float4 **exact, const float4 **pre,
                           float **keepRaw = nullptr)
{
    if (keepRaw) *keepRaw = nullptr;
    int rc;
    *exact = nullptr;
    if (pre) *pre = nullptr;
    if ((rc = uploadWith<float4>(ctx, s, 3 * n, exact, [](float4 *) {}, true)) != RTB_OK) return rc; // allocations (zeroed)
    if (pre && (rc = uploadWith<float4>(ctx, s, 3 * n, pre, [](float4 *) {}, true)) != RTB_OK) return rc;
    if (n == 0) return RTB_OK;
    char *st = nullptr;
    if ((rc = stageFill(ctx, n * 12 * sizeof(float), &st, [&](char *dst) { memcpy(dst, host, n * 12 * sizeof(float)); }, host, &s->direct_sources)) != RTB_OK) return rc;
    void *raw = nullptr;
    CUDA_TRY(ctx, cudaMallocAsync(&raw, n * 12 * sizeof(float), ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(raw, st, n * 12 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    s->h2d_bytes += (int64_t)(n * 12 * sizeof(float));
    k_pack_triangles<<<(unsigned int)((n + 255) / 256), 256, 0, ctx->stream>>>((const float *)raw, (int)n, const_cast<float4 *>(*exact),
                                                                             pre ? const_cast<float4 *>(*pre) : nullptr);
    CUDA_TRY(ctx, cudaGetLastError());
    if (keepRaw) *keepRaw = (float *)raw;
    else CUDA_TRY(ctx, cudaFreeAsync(raw, ctx->stream));
    return RTB_OK;
}

// Pair stream (DScene::pre2): the rejection-test records of list positions 2p and 2p + 1, interleaved component by
// component so that the 128-bit loads of the scan deliver 64-bit register pairs for the packed FP32 instructions.
// One thread per list position; the unused half of a trailing odd pair is zero (allocation is cleared).
__global__ void k_pack_pairs(const uint32_t *__restrict__ refs, unsigned int n_refs, const float4 *__restrict__ tri_pre,
                             float *__restrict__ pre2)
{
    const unsigned int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_refs) return;
    const float4 *src = tri_pre + 3ull * refs[j];
    const float4 q0 = src[0], q1 = src[1], q2 = src[2]; // {a.xyz, A1e} {e1.xyz, Ee} {e2.xyz, 0}
    float *dst = pre2 + 24ull * (j >> 1) + (j & 1u);
    dst[0] = q0.x; dst[2] = q0.y; dst[4] = q0.z; dst[6] = q0.w;
    dst[8] = q1.x; dst[10] = q1.y; dst[12] = q1.z; dst[14] = q1.w;
    dst[16] = q2.x; dst[18] = q2.y; dst[20] = q2.z; dst[22] = 0.f;
}

// builds DScene::pre2 for the reference array `refs` (device) -- queued behind the copies / kernels that produce it
static int packPairs(rtb_ctx *ctx, rtb_scene *s, const uint32_t *refs, size_t n_refs)
{
    const size_t pairs = (n_refs + 1) / 2;
    int rc = uploadWith<float4>(ctx, s, 6 * pairs, &s->d.pre2, [](float4 *) {}, true); // zero-filled allocation
    if (rc != RTB_OK || n_refs == 0) return rc;
    k_pack_pairs<<<(unsigned int)((n_refs + 255) / 256), 256, 0, ctx->stream>>>(refs, (unsigned int)n_refs, s->d.tri_pre,
                                                                                reinterpret_cast<float *>(const_cast<float4 *>(s->d.pre2)));
    CUDA_TRY(ctx, cudaGetLastError());
    return RTB_OK;
}

template <class T> static int deviceArray(rtb_ctx *ctx, rtb_scene *s, size_t n, T **dev, bool keep)
{
    void *p = nullptr;
    CUDA_TRY(ctx, cudaMallocAsync(&p, (n ? n : 1) * sizeof(T), ctx->stream));
    if (keep) { s->allocs.push_back(p); s->bytes += (int64_t)(n * sizeof(T)); }
    *dev = (T *)p;
    return RTB_OK;
}

// The k-d arrays the kernels walk: every leaf list on an even position of the reference array (k_kd_pad_sizes / k_kd_relayout,
// rtb_misc.cuh), then the pair stream over that array.  `padded_refs` = sum of the leaves' padded list lengths (exact, or an
// upper bound).  RTB_KD_PAD=0: the arrays as they came.
static int padKdLists(rtb_ctx *ctx, rtb_scene *s, long long padded_refs)
{
    DScene &d = s->d;
    s->kd_nodes_plain = d.kd_nodes; s->kd_tris_plain = d.kd_tris;
    static const bool on = !(getenv("RTB_KD_PAD") && atoi(getenv("RTB_KD_PAD")) == 0);
    const long long n = s->kd_nodes;
    // (leaves that share or overlap lists could blow the copy up: such a tree keeps its layout)
    if (!on || n <= 0 || padded_refs <= 0 || padded_refs > 2 * (s->kd_refs + n) + 64 || padded_refs > 0x7fffffffLL)
        return packPairs(ctx, s, d.kd_tris, (size_t)s->kd_refs);
    cudaStream_t st = ctx->stream;
    unsigned int *d_size = nullptr, *d_first = nullptr;
    void *d_tmp = nullptr;
    uint2 *nodes_out = nullptr;
    uint32_t *refs_out = nullptr;
    auto cleanup = [&]() { if (d_size) cudaFreeAsync(d_size, st); if (d_first) cudaFreeAsync(d_first, st); if (d_tmp) cudaFreeAsync(d_tmp, st); };
#define PAD_TRY(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); return fail(ctx, RTB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } } while (0)
    PAD_TRY(cudaMallocAsync((void **)&d_size, (size_t)(n + 1) * sizeof(unsigned int), st));
    PAD_TRY(cudaMallocAsync((void **)&d_first, (size_t)(n + 1) * sizeof(unsigned int), st));
    k_kd_pad_sizes<<<(unsigned int)((n + 1 + 255) / 256), 256, 0, st>>>(d.kd_nodes, (int)n, d_size);
    size_t need = 0;
    PAD_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, d_size, d_first, (int)n + 1, st));
    PAD_TRY(cudaMallocAsync(&d_tmp, need ? need : 1, st));
    PAD_TRY(cub::DeviceScan::ExclusiveSum(d_tmp, need, d_size, d_first, (int)n + 1, st));
    int rc;
    if ((rc = deviceArray(ctx, s, (size_t)n, &nodes_out, true)) != RTB_OK || (rc = deviceArray(ctx, s, (size_t)padded_refs, &refs_out, true)) != RTB_OK) { cleanup(); return rc; }
    PAD_TRY(cudaMemsetAsync(refs_out, 0, (size_t)padded_refs * sizeof(uint32_t), st));
    k_kd_relayout<<<(unsigned int)((n + 255) / 256), 256, 0, st>>>(d.kd_nodes, (int)n, d_first, d.kd_tris, nodes_out, refs_out, (unsigned int)padded_refs);
    PAD_TRY(cudaGetLastError());
#undef PAD_TRY
    cleanup();
    d.kd_nodes = nodes_out; d.kd_tris = refs_out;
    return packPairs(ctx, s, refs_out, (size_t)padded_refs);
}

// sum of the leaves' padded list lengths of a caller's tree (the validation tasks of rtb_scene_upload compute it on the side;
// uploads that skip them -- the replicas of an rtb_multi_scene_upload -- take this pass)
static long long paddedKdRefs(const rtb_flat_scene *f)
{
    long long total = 0;
    for (int i = 0; i < f->n_kd_nodes; i++)
        total += ((f->kd_nodes[i].b & 3u) == 3u) ? (long long)(((f->kd_nodes[i].b >> 2) + 1u) & ~1u) : 0;
    return total;
}

// pre-order k-d array -> 0 when it is a well-formed tree (every inner node's right child lies behind its left
// subtree, every node reached exactly once), maxDepth = deepest node.  One linear pass with an explicit stack of
// pending right children: the recursive walk took 0.2 ms of every upload.
// (range form: is nodes[a .. b) a well-formed subtree that ends exactly at b, its root at depth `depth0`?  A well-formed pre-order
// array consists of such ranges -- node 0's left subtree [1, right) and right subtree [right, n), and so on down -- which is how
// rtb_scene_upload cuts the check into tasks for its worker threads.)
static int kdDepthRange(const rtb_kdnode *nodes, int a, int b, int depth0, int &maxDepth)
{
    // Pending right children, innermost last, with the depth they resume at; slot 0 is a sentinel, "the range ends at b".
    // Whether a node is a leaf is a coin toss for the branch predictor (69 k nodes: 0.45 ms of every upload with a branch per
    // node and a std::vector stack), so the pass is written with selects: both outcomes are computed, the slot above the top is
    // written either way and only an inner node keeps it.  Invariant: pending entries <= depth - depth0 <= 64, so 72 slots suffice.
    maxDepth = depth0;
    if (b <= a) return -1;
    int pendR[72], pendD[72];
    pendR[0] = b; pendD[0] = depth0;
    int sp = 0, depth = depth0, deepest = depth0;
    unsigned int bad = 0;
    for (int i = a; i < b; i++)
    {
        const unsigned int w = nodes[i].b;
        const bool leaf = (w & 3u) == 3u;
        const int right = (int)(w >> 2);
        const int top = pendR[sp];
        deepest = depth > deepest ? depth : deepest;
        // leaf: the next node in pre-order is the nearest pending right child (the sentinel: the end of the range);
        // inner: its right child lies behind its left child and before the enclosing pending right child
        const unsigned int badLeaf = (unsigned int)(top != i + 1), badInner = (unsigned int)(right <= i + 1) | (unsigned int)(right >= top);
        bad |= leaf ? badLeaf : badInner;
        pendR[sp + 1] = right;
        pendD[sp + 1] = depth + 1;
        const int resume = pendD[sp];
        depth = leaf ? resume : depth + 1;
        sp += leaf ? -1 : 1;
        if ((sp < 0) | (depth > 64)) break; // the subtree has closed (at b - 1, or `bad` is set) / deeper than any supported tree
    }
    maxDepth = deepest;
    return (!bad && sp == -1 && depth <= 64) ? 0 : -1; // sp >= 0: ran out of nodes with subtrees still open
}

// nodes[0 .. n) cut into up to 8 subtree ranges, largest split first; the nodes split at are checked here (inner, right child
// inside the range).  A range whose root cannot be split stays whole: its own kdDepthRange reports what is wrong with it.
struct KdRange { int a, b, depth; };
static std::vector<KdRange> kdSubtrees(const rtb_kdnode *nodes, int n)
{
    std::vector<KdRange> ranges(1, KdRange{0, n, 0});
    std::vector<char> whole(1, 0);
    while (ranges.size() < 8)
    {
        int k = -1;
        for (size_t i = 0; i < ranges.size(); i++)
            if (!whole[i] && ranges[i].b - ranges[i].a >= 64 && (k < 0 || ranges[i].b - ranges[i].a > ranges[(size_t)k].b - ranges[(size_t)k].a)) k = (int)i;
        if (k < 0) break;
        const KdRange r = ranges[(size_t)k];
        const unsigned int w = nodes[r.a].b;
        const int right = (int)(w >> 2);
        if ((w & 3u) == 3u || right <= r.a + 1 || right >= r.b) { whole[(size_t)k] = 1; continue; }
        ranges[(size_t)k] = KdRange{r.a + 1, right, r.depth + 1};
        ranges.push_back(KdRange{right, r.b, r.depth + 1});
        whole.push_back(0);
    }
    return ranges;
}

extern "C" int rtb_kd_validate(const rtb_kdnode *nodes, int32_t n, int32_t *max_depth)
{
    if (!nodes || n <= 0) return RTB_ERR_INVALID;
    int deepest = 0; // the same decomposition rtb_scene_upload hands to its checker threads, here one range after the other
    for (const KdRange &r : kdSubtrees(nodes, n))
    {
        int depth = 0;
        if (kdDepthRange(nodes, r.a, r.b, r.depth, depth) != 0) return RTB_ERR_INVALID;
        deepest = depth > deepest ? depth : deepest;
    }
    if (max_depth) *max_depth = deepest;
    return RTB_OK;
}



// ---- grid built on the device (rtb_build_grid.cuh) ------------------------------------------------------------
static int buildGridOnDevice(rtb_ctx *ctx, rtb_scene *s, const rtb_flat_scene *f, float *d_raw)
{
    DScene &d = s->d;
    const int n = f->n_tris, R = f->grid_build_resolution;
    cudaStream_t st = ctx->stream;
    std::vector<void *> temps;
    auto temp = [&](size_t bytes, void **p) { cudaError_t e = cudaMallocAsync(p, bytes ? bytes : 1, st); if (e == cudaSuccess) temps.push_back(*p); return e; };
    auto cleanup = [&]() { for (void *p : temps) cudaFreeAsync(p, st); };
#define GRID_TRY(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); return fail(ctx, RTB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } } while (0)
    float *d_bounds = nullptr; // d_raw: the raw triangle records already on the device (uploadTriangles)
    GRID_TRY(temp(6 * sizeof(float), (void **)&d_bounds));
    const float init[6] = {FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX};
    GRID_TRY(cudaMemcpyAsync(d_bounds, init, sizeof(init), cudaMemcpyHostToDevice, st));
    k_grid_bounds<<<148, 256, 0, st>>>(d_raw, n, d_bounds);
    float b[6];
    GRID_TRY(cudaMemcpyAsync(b, d_bounds, sizeof(b), cudaMemcpyDeviceToHost, st));
    GRID_TRY(cudaStreamSynchronize(st));

    // sizing with the reference's float expressions (Tunnel.cpp:372-404)
    GridSizing G;
    G.exact = f->grid_build_exact ? 1 : 0;
    const float width = b[3] - b[0], height = b[4] - b[1], depth = b[5] - b[2];
    if (f->accel == RTB_ACCEL_REGULAR_GRID)
    {
        const float maxLength = std::max(std::max(width, height), depth);
        const float size = maxLength / (R - 1);
        for (int a = 0; a < 3; a++) { G.cell[a] = size; G.origin[a] = b[a] - size / 2; }
        G.dims[0] = (int)(width / size + 1.5f); G.dims[1] = (int)(height / size + 1.5f); G.dims[2] = (int)(depth / size + 1.5f);
    }
    else
    {
        G.cell[0] = width / (R - 1); G.cell[1] = height / (R - 1); G.cell[2] = depth / (R - 1);
        for (int a = 0; a < 3; a++) { G.origin[a] = b[a] - G.cell[a] / 2; G.dims[a] = R; }
    }
    const int64_t cells = (int64_t)G.dims[0] * G.dims[1] * G.dims[2];
    if (G.dims[0] <= 0 || G.dims[1] <= 0 || G.dims[2] <= 0 || cells > 0x7fffffffLL || !(G.cell[0] > 0) || !(G.cell[1] > 0) || !(G.cell[2] > 0))
    {
        cleanup();
        return fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: degenerate tunnel bounds, cannot size the grid");
    }
    const int64_t nWords = (cells + 31) / 32;

    // count -> scan -> emit -> sort
    unsigned int *d_count = nullptr, *d_offset = nullptr;
    GRID_TRY(temp((size_t)(n + 1) * sizeof(unsigned int), (void **)&d_count));
    GRID_TRY(temp((size_t)(n + 1) * sizeof(unsigned int), (void **)&d_offset));
    GRID_TRY(cudaMemsetAsync(d_count, 0, (size_t)(n + 1) * sizeof(unsigned int), st));
    const int tb = 256, nb = (n + tb - 1) / tb;
    k_grid_count<<<nb, tb, 0, st>>>(d_raw, n, G, d_count);
    void *d_tmp = nullptr;
    size_t tmpBytes = 0, need = 0;
    GRID_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, d_count, d_offset, n + 1, st));
    tmpBytes = need;
    GRID_TRY(temp(tmpBytes, &d_tmp));
    GRID_TRY(cub::DeviceScan::ExclusiveSum(d_tmp, tmpBytes, d_count, d_offset, n + 1, st));
    unsigned int total = 0;
    GRID_TRY(cudaMemcpyAsync(&total, d_offset + n, sizeof(total), cudaMemcpyDeviceToHost, st));
    GRID_TRY(cudaStreamSynchronize(st));
    if (total == 0 || total > 0x7fffffffu) { cleanup(); return fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: grid reference count out of range"); }
    unsigned long long *d_keys = nullptr, *d_sorted = nullptr;
    GRID_TRY(temp((size_t)total * sizeof(unsigned long long), (void **)&d_keys));
    GRID_TRY(temp((size_t)total * sizeof(unsigned long long), (void **)&d_sorted));
    k_grid_emit<<<nb, tb, 0, st>>>(d_raw, n, G, d_offset, d_keys);
    int cellBits = 1;
    while ((1ll << cellBits) < cells) cellBits++;
    void *d_tmp2 = nullptr;
    GRID_TRY(cub::DeviceRadixSort::SortKeys(nullptr, need, d_keys, d_sorted, (int)total, 0, 32 + cellBits, st));
    GRID_TRY(temp(need, &d_tmp2));
    GRID_TRY(cub::DeviceRadixSort::SortKeys(d_tmp2, need, d_keys, d_sorted, (int)total, 0, 32 + cellBits, st));

    // directory
    uint2 *d_words = nullptr;
    uint32_t *d_cell_tris = nullptr, *d_cell_start = nullptr;
    int rc;
    if ((rc = deviceArray(ctx, s, (size_t)nWords, &d_words, true)) != RTB_OK) { cleanup(); return rc; }
    if ((rc = deviceArray(ctx, s, (size_t)total, &d_cell_tris, true)) != RTB_OK) { cleanup(); return rc; }
    GRID_TRY(cudaMemsetAsync(d_words, 0, (size_t)nWords * sizeof(uint2), st));
    unsigned int *d_head = nullptr, *d_rank = nullptr;
    GRID_TRY(temp((size_t)(total + 1) * sizeof(unsigned int), (void **)&d_head));
    GRID_TRY(temp((size_t)(total + 1) * sizeof(unsigned int), (void **)&d_rank));
    GRID_TRY(cudaMemsetAsync(d_head + total, 0, sizeof(unsigned int), st));
    const unsigned int eb = (total + tb - 1) / tb;
    k_grid_heads<<<eb, tb, 0, st>>>(d_sorted, total, d_cell_tris, d_head, d_words);
    void *d_tmp3 = nullptr;
    GRID_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, d_head, d_rank, (int)total + 1, st));
    GRID_TRY(temp(need, &d_tmp3));
    GRID_TRY(cub::DeviceScan::ExclusiveSum(d_tmp3, need, d_head, d_rank, (int)total + 1, st));
    unsigned int nRuns = 0;
    GRID_TRY(cudaMemcpyAsync(&nRuns, d_rank + total, sizeof(nRuns), cudaMemcpyDeviceToHost, st));
    GRID_TRY(cudaStreamSynchronize(st));
    if ((rc = deviceArray(ctx, s, (size_t)nRuns + 1, &d_cell_start, true)) != RTB_OK) { cleanup(); return rc; }
    k_grid_starts<<<eb, tb, 0, st>>>(d_head, d_rank, total, d_cell_start, nRuns);
    unsigned int *d_pop = nullptr, *d_wrank = nullptr;
    GRID_TRY(temp((size_t)nWords * sizeof(unsigned int), (void **)&d_pop));
    GRID_TRY(temp((size_t)nWords * sizeof(unsigned int), (void **)&d_wrank));
    const unsigned int wb = (unsigned int)((nWords + tb - 1) / tb);
    k_grid_word_pop<<<wb, tb, 0, st>>>(d_words, nWords, d_pop);
    void *d_tmp4 = nullptr;
    GRID_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, d_pop, d_wrank, (int)nWords, st));
    GRID_TRY(temp(need, &d_tmp4));
    GRID_TRY(cub::DeviceScan::ExclusiveSum(d_tmp4, need, d_pop, d_wrank, (int)nWords, st));
    k_grid_word_rank<<<wb, tb, 0, st>>>(d_words, nWords, d_wrank);
    GRID_TRY(cudaGetLastError());
    cleanup();
    GRID_TRY(cudaStreamSynchronize(st));
#undef GRID_TRY

    d.g_origin = {G.origin[0], G.origin[1], G.origin[2]};
    d.g_cell = {G.cell[0], G.cell[1], G.cell[2]};
    d.nx = G.dims[0]; d.ny = G.dims[1]; d.nz = G.dims[2];
    d.g_extent = {d.g_cell.x * d.nx, d.g_cell.y * d.ny, d.g_cell.z * d.nz};
    d.g_far = {d.g_origin.x + d.g_extent.x, d.g_origin.y + d.g_extent.y, d.g_origin.z + d.g_extent.z};
    d.g_words = d_words; d.g_start = d_cell_start; d.g_tris = d_cell_tris;
    s->grid_cells_used = nRuns; s->grid_refs = total; s->grid_words = nWords;
    return packPairs(ctx, s, d_cell_tris, (size_t)total);
}

// ---- SAH k-d tree built on the device (rtb_build_kd.cuh) -------------------------------------------------------
static int buildKdOnDevice(rtb_ctx *ctx, rtb_scene *s, const rtb_flat_scene *f, float *d_raw)
{
    DScene &d = s->d;
    const int n = f->n_tris, leafSize = f->kd_build_leaf_size > 0 ? f->kd_build_leaf_size : 8, maxDepth = f->kd_build_max_depth;
    const int N = f->kd_build_candidates > 0 ? f->kd_build_candidates : 100;
    if (N < 2 || N > RTB_KDB_MAX_CAND) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: kd_build_candidates must be in [2, 128]");
    if (2 * (maxDepth + 1) + 2 >= RTB_KD_STACK || maxDepth + 2 > RTB_KDB_MAX_LEVELS)
        return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scene_upload: kd_build_max_depth too deep for the 50-entry traversal stack");
    cudaStream_t st = ctx->stream;
    std::vector<void *> temps;
    auto temp = [&](size_t bytes, void **p) { cudaError_t e = cudaMallocAsync(p, bytes ? bytes : 1, st); if (e == cudaSuccess) temps.push_back(*p); return e; };
    auto cleanup = [&]() { for (void *p : temps) cudaFreeAsync(p, st); };
#define KD_TRY(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); return fail(ctx, RTB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } } while (0)
    float *d_bounds = nullptr, *d_lo = nullptr, *d_hi = nullptr; // d_raw: the raw triangle records already on the device
    KD_TRY(temp(6 * sizeof(float), (void **)&d_bounds));
    const float init[6] = {FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX};
    KD_TRY(cudaMemcpyAsync(d_bounds, init, sizeof(init), cudaMemcpyHostToDevice, st));
    k_grid_bounds<<<148, 256, 0, st>>>(d_raw, n, d_bounds); // root box = bounds of all vertices (Tunnel.cpp:486-510)
    KD_TRY(temp((size_t)3 * n * sizeof(float), (void **)&d_lo));
    KD_TRY(temp((size_t)3 * n * sizeof(float), (void **)&d_hi));
    const int tb = 256, nb = (n + tb - 1) / tb;
    k_kd_extents<<<nb, tb, 0, st>>>(d_raw, n, d_lo, d_hi);

    size_t nodeCap = (size_t)n * 2 + 1024;
    KdBuildNode *d_nodes = nullptr;
    KD_TRY(temp(nodeCap * sizeof(KdBuildNode), (void **)&d_nodes));
    uint32_t *d_refs = nullptr;
    KD_TRY(temp((size_t)n * sizeof(uint32_t), (void **)&d_refs));
    k_kd_root<<<nb, tb, 0, st>>>(d_nodes, d_bounds, n, d_refs);
    int *d_totals = nullptr;
    KD_TRY(temp(4 * sizeof(int), (void **)&d_totals));

    KdLeafChunks chunks;
    memset(&chunks, 0, sizeof(chunks));
    std::vector<int> levelFirst, levelCount;
    int first = 0, count = 1, totalNodes = 1;
    for (int level = 0; count > 0; level++)
    {
        if (level >= RTB_KDB_MAX_LEVELS) { cleanup(); return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scene_upload: k-d build exceeded the level limit"); }
        levelFirst.push_back(first); levelCount.push_back(count);
        int *d_childOff = nullptr, *d_leafOff = nullptr, *d_innerRank = nullptr;
        KD_TRY(temp((size_t)count * sizeof(int), (void **)&d_childOff));
        KD_TRY(temp((size_t)count * sizeof(int), (void **)&d_leafOff));
        KD_TRY(temp((size_t)count * sizeof(int), (void **)&d_innerRank));
        k_kd_eval<<<count, RTB_KDB_THREADS, 0, st>>>(d_nodes, first, d_refs, d_lo, d_hi, n, leafSize, maxDepth, N);
        k_kd_level_scan<<<1, 1024, 0, st>>>(d_nodes, first, count, d_childOff, d_leafOff, d_innerRank, d_totals);
        int totals[3] = {0, 0, 0};
        KD_TRY(cudaMemcpyAsync(totals, d_totals, sizeof(totals), cudaMemcpyDeviceToHost, st));
        KD_TRY(cudaStreamSynchronize(st));
        const int nextRefs = totals[0], leafRefs = totals[1], inner = totals[2];
        if (nextRefs < 0 || leafRefs < 0) { cleanup(); return fail(ctx, RTB_ERR_OOM, "rtb_scene_upload: k-d build reference count overflow"); }
        if ((size_t)totalNodes + 2 * (size_t)inner > nodeCap)
        { // grow the node table (level order: the children of this level follow everything built so far)
            const size_t cap = ((size_t)totalNodes + 2 * (size_t)inner) * 2;
            KdBuildNode *bigger = nullptr;
            KD_TRY(temp(cap * sizeof(KdBuildNode), (void **)&bigger));
            KD_TRY(cudaMemcpyAsync(bigger, d_nodes, (size_t)totalNodes * sizeof(KdBuildNode), cudaMemcpyDeviceToDevice, st));
            d_nodes = bigger; nodeCap = cap;
        }
        uint32_t *d_next = nullptr, *d_chunk = nullptr;
        KD_TRY(temp((size_t)nextRefs * sizeof(uint32_t), (void **)&d_next));
        KD_TRY(temp((size_t)leafRefs * sizeof(uint32_t), (void **)&d_chunk));
        chunks.p[level] = d_chunk;
        k_kd_partition<<<count, RTB_KDB_THREADS, 0, st>>>(d_nodes, first, level, totalNodes, d_refs, d_next, d_chunk, d_childOff, d_leafOff,
                                                          d_innerRank, d_lo, d_hi, n);
        KD_TRY(cudaGetLastError());
        d_refs = d_next;
        first = totalNodes; count = 2 * inner; totalNodes += 2 * inner;
    }
    const int levels = (int)levelFirst.size();
    for (int l = levels - 1; l >= 0; l--) k_kd_sizes<<<(levelCount[l] + 255) / 256, 256, 0, st>>>(d_nodes, levelFirst[l], levelCount[l]);
    for (int l = 0; l < levels; l++) k_kd_place<<<(levelCount[l] + 255) / 256, 256, 0, st>>>(d_nodes, levelFirst[l], levelCount[l]);
    KdBuildNode root;
    float b[6];
    KD_TRY(cudaMemcpyAsync(&root, d_nodes, sizeof(root), cudaMemcpyDeviceToHost, st));
    KD_TRY(cudaMemcpyAsync(b, d_bounds, sizeof(b), cudaMemcpyDeviceToHost, st));
    KD_TRY(cudaStreamSynchronize(st));
    if (root.subNodes != totalNodes) { cleanup(); return fail(ctx, RTB_ERR_CUDA, "rtb_scene_upload: k-d build inconsistent (subtree sizes)"); }
    uint2 *d_out = nullptr;
    uint32_t *d_leaf = nullptr;
    int rc;
    if ((rc = deviceArray(ctx, s, (size_t)totalNodes, &d_out, true)) != RTB_OK) { cleanup(); return rc; }
    if ((rc = deviceArray(ctx, s, (size_t)root.subRefs, &d_leaf, true)) != RTB_OK) { cleanup(); return rc; }
    k_kd_emit<<<(totalNodes + 255) / 256, 256, 0, st>>>(d_nodes, totalNodes, chunks, d_out, d_leaf);
    KD_TRY(cudaGetLastError());
    cleanup();
#undef KD_TRY
    d.kd_min = {b[0], b[1], b[2]};
    d.kd_size = {b[3] - b[0], b[4] - b[1], b[5] - b[2]}; // Grid(near, far): size = far - near (Grid.cpp:13-17)
    d.kd_nodes = d_out; d.kd_tris = d_leaf;
    s->kd_nodes = totalNodes; s->kd_refs = root.subRefs; s->kd_levels = levels;
    return padKdLists(ctx, s, (long long)root.subRefs + ((long long)totalNodes + 1) / 2); // disjoint lists, at most one padding slot per leaf
}

// Index / structure checks of rtb_scene_upload that scan whole streams (k-d nodes, leaf and cell references: 0.6 ms
// of a 1 ms upload on the host) run on worker threads while the calling thread stages and queues the copies.  The
// verdict is collected before anything that indexes with those streams is launched (k_pack_pairs, the renders); the
// copies and k_pack_triangles do not index.
struct BackgroundChecks
{
    typedef std::function<std::pair<int, const char *>()> Task; // -> {code, message}
    WorkerPool *pool = nullptr;
    std::vector<Task> tasks;
    std::mutex m;
    int code = RTB_OK;
    std::string msg;
    bool enabled = true; // false: the caller has validated this very flat scene already (rtb_multi_scene_upload: replicas)
    bool started = false;
    std::atomic<long long> kd_padded{0}; // by-product of the k-d leaf checks: sum of the padded list lengths (padKdLists)
    void keep(const std::pair<int, const char *> &r)
    {
        if (r.first == RTB_OK) return;
        std::lock_guard<std::mutex> lock(m);
        if (code == RTB_OK) { code = r.first; msg = r.second; }
    }
    template <class Fn> void run(Fn fn) { if (enabled) tasks.emplace_back(fn); } // queued; start() hands the tasks to the pool
    void start()
    {
        if (!enabled || started || tasks.empty() || !pool || pool->workers() == 0) return;
        started = true;
        const size_t W = (size_t)pool->workers();
        pool->begin([this, W](int w) { for (size_t t = (size_t)w - 1; t < tasks.size(); t += W) keep(tasks[t]()); });
    }
    void join() // a failure is kept in code / msg
    {
        if (started) pool->finish();
        else for (Task &t : tasks) keep(t()); // never handed to the pool: here and now
        started = false;
        tasks.clear();
    }
    ~BackgroundChecks() { join(); }
};

static bool gridHeaderOk(const rtb_flat_scene *f)
{
    const int64_t cells = (int64_t)f->grid_dims[0] * f->grid_dims[1] * f->grid_dims[2];
    return !(f->grid_dims[0] <= 0 || f->grid_dims[1] <= 0 || f->grid_dims[2] <= 0 || cells > 0x7fffffffLL ||
             f->n_cellwords != (cells + 31) / 32 || !f->grid_words || !f->grid_cell_start || (f->n_cell_refs > 0 && !f->grid_cell_tris));
}
static bool kdHeaderOk(const rtb_flat_scene *f) { return !(f->n_kd_nodes <= 0 || !f->kd_nodes || (f->n_kd_refs > 0 && !f->kd_leaf_tris)); }

// The whole-stream checks of the accelerator arrays the walks index with, cut into tasks of similar size for the context's
// checker threads (nothing is queued when the header fields are inconsistent: sceneUpload refuses such a scene before anything
// reads its arrays).  Every condition is local -- a word's rank against the next word's, a list start against the next, a
// reference against the triangle count -- except the shape of the k-d tree, which splits into subtrees (kdDepthRange).
static void queueSceneChecks(const rtb_flat_scene *f, BackgroundChecks &checks)
{
    typedef std::pair<int, const char *> R;
    const int64_t CHUNKS = 4;
    auto slices = [&](int64_t n, const std::function<R(int64_t, int64_t)> &body) { // body(lo, hi) over [0, n) in CHUNKS slices
        for (int64_t c = 0; c < CHUNKS; c++)
        {
            const int64_t lo = n * c / CHUNKS, hi = n * (c + 1) / CHUNKS;
            if (hi > lo) checks.run([body, lo, hi]() { return body(lo, hi); });
        }
    };
    if (f->n_tris < 0) return;
    const uint32_t nTris = (uint32_t)f->n_tris;
    if ((f->accel == RTB_ACCEL_REGULAR_GRID || f->accel == RTB_ACCEL_FLAT_GRID) && f->grid_words)
    {
        if (!gridHeaderOk(f)) return;
        if (f->n_cells_used < 0) { checks.run([]() { return R((int)RTB_ERR_INVALID, "rtb_scene_upload: negative cell count"); }); return; }
        // the directory the walks index with: every word's rank is the number of occupied cells before it, the occupied
        // cells number n_cells_used, and the list starts ascend from 0 to n_cell_refs (no empty list: the pair scan needs
        // at least one entry)
        slices(f->n_cellwords, [f](int64_t lo, int64_t hi) {
            bool bad = lo == 0 && f->grid_words[0].rank != 0;
            for (int64_t w = lo; w < hi; w++)
            {
                const uint64_t next = w + 1 < f->n_cellwords ? (uint64_t)f->grid_words[w + 1].rank : (uint64_t)f->n_cells_used;
                bad |= (uint64_t)f->grid_words[w].rank + (uint64_t)__builtin_popcount(f->grid_words[w].bits) != next;
            }
            return R(bad ? (int)RTB_ERR_INVALID : (int)RTB_OK, "rtb_scene_upload: grid word ranks do not match the occupancy bits");
        });
        checks.run([f]() {
            const int64_t cells = (int64_t)f->grid_dims[0] * f->grid_dims[1] * f->grid_dims[2];
            if (f->n_cellwords == 0 && f->n_cells_used != 0) return R((int)RTB_ERR_INVALID, "rtb_scene_upload: grid word ranks do not match the occupancy bits");
            if (f->n_cellwords > 0 && (cells & 31) != 0 && (f->grid_words[f->n_cellwords - 1].bits >> (cells & 31)) != 0)
                return R((int)RTB_ERR_INVALID, "rtb_scene_upload: occupancy bits beyond the last cell");
            const bool ends = f->grid_cell_start[0] == 0 && (int64_t)f->grid_cell_start[f->n_cells_used] == f->n_cell_refs;
            return R(ends ? (int)RTB_OK : (int)RTB_ERR_INVALID, "rtb_scene_upload: grid cell list starts are not strictly ascending from 0 to n_cell_refs");
        });
        slices(f->n_cells_used, [f](int64_t lo, int64_t hi) {
            bool order = true;
            for (int64_t i = lo; i < hi; i++) order &= f->grid_cell_start[i] < f->grid_cell_start[i + 1];
            return R(order ? (int)RTB_OK : (int)RTB_ERR_INVALID, "rtb_scene_upload: grid cell list starts are not strictly ascending from 0 to n_cell_refs");
        });
        slices(f->n_cell_refs, [f, nTris](int64_t lo, int64_t hi) {
            uint32_t maxRef = 0; // branch-free maximum: the compiler vectorises it (up to 6.4 M references)
            for (int64_t i = lo; i < hi; i++) maxRef = f->grid_cell_tris[i] > maxRef ? f->grid_cell_tris[i] : maxRef;
            return R(maxRef >= nTris ? (int)RTB_ERR_INVALID : (int)RTB_OK, "rtb_scene_upload: grid triangle reference out of range");
        });
    }
    else if ((f->accel == RTB_ACCEL_KD_MEDIAN || f->accel == RTB_ACCEL_KD_SAH) && f->kd_nodes)
    {
        if (!kdHeaderOk(f)) return;
        // the tree's shape: one task per subtree range
        for (const KdRange &r : kdSubtrees(f->kd_nodes, f->n_kd_nodes))
            checks.run([f, r]() {
                int maxDepth = 0;
                if (kdDepthRange(f->kd_nodes, r.a, r.b, r.depth, maxDepth) != 0) return R((int)RTB_ERR_INVALID, "rtb_scene_upload: k-d nodes are not a pre-order tree");
                if (2 * maxDepth + 2 >= RTB_KD_STACK)
                    return R((int)RTB_ERR_UNSUPPORTED, "rtb_scene_upload: k-d tree deeper than the 50-entry traversal stack allows");
                return R((int)RTB_OK, "");
            });
        std::atomic<long long> *padded = &checks.kd_padded;
        slices(f->n_kd_nodes, [f, padded](int64_t lo, int64_t hi) { // branch-free maxima (the compiler vectorises them)
            int64_t leafEnd = 0;
            long long pad = 0;
            for (int64_t i = lo; i < hi; i++)
            {
                const bool leaf = (f->kd_nodes[i].b & 3u) == 3u;
                const int64_t e = leaf ? (int64_t)f->kd_nodes[i].a + (f->kd_nodes[i].b >> 2) : 0;
                leafEnd = e > leafEnd ? e : leafEnd;
                pad += leaf ? (long long)(((f->kd_nodes[i].b >> 2) + 1u) & ~1u) : 0;
            }
            padded->fetch_add(pad, std::memory_order_relaxed);
            return R(leafEnd > f->n_kd_refs ? (int)RTB_ERR_INVALID : (int)RTB_OK, "rtb_scene_upload: k-d leaf range out of bounds");
        });
        slices(f->n_kd_refs, [f, nTris](int64_t lo, int64_t hi) {
            uint32_t maxRef = 0;
            for (int64_t i = lo; i < hi; i++) maxRef = f->kd_leaf_tris[i] > maxRef ? f->kd_leaf_tris[i] : maxRef;
            return R(maxRef >= nTris ? (int)RTB_ERR_INVALID : (int)RTB_OK, "rtb_scene_upload: k-d triangle reference out of range");
        });
    }
}

// RTB_UPLOAD_TIMING=1: host-side laps of rtb_scene_upload on stderr (profiling aid)
struct UploadLaps
{
    bool on;
    std::chrono::steady_clock::time_point t0;
    std::string text;
    UploadLaps() : on(getenv("RTB_UPLOAD_TIMING") && atoi(getenv("RTB_UPLOAD_TIMING"))), t0(std::chrono::steady_clock::now()) {}
    void lap(const char *what)
    {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        char buf[64];
        snprintf(buf, sizeof(buf), " %s %.0f us;", what, std::chrono::duration<double, std::micro>(t1 - t0).count());
        text += buf;
        t0 = t1;
    }
    ~UploadLaps() { if (on) fprintf(stderr, "rtb_scene_upload:%s\n", text.c_str()); }
};

// The verdict of the whole-stream checks, before anything indexes with the checked streams.  Within an rtb_multi_scene_upload
// the producer publishes it and the replicas (which skipped the checks) wait for it here.
static int collectVerdict(rtb_ctx *ctx, BackgroundChecks &checks)
{
    checks.join();
    if (checks.code != RTB_OK) return fail(ctx, checks.code, checks.msg);
    if (StageShare *sh = ctx->share)
    {
        if (ctx->share_producer) sh->verdict.store(1, std::memory_order_release);
        else if (!sh->waitVerdict()) return fail(ctx, RTB_ERR_INVALID, "rtb_multi_scene_upload: the first device's upload failed");
    }
    return RTB_OK;
}

// upper bound of the bytes one upload of `f` stages (every stream rounded up to the ring's 256-byte granules)
static size_t stagedBytesBound(const rtb_flat_scene *f)
{
    auto r = [](double n, size_t elem) { return n > 0 ? (((size_t)n * elem + 255) & ~(size_t)255) : (size_t)0; };
    size_t t = r(f->loose_tri ? f->n_loose : 0, 48) + r(f->tri ? f->n_tris : 0, 48) + r(f->tri_material ? f->n_tris : 0, 4);
    if ((f->accel == RTB_ACCEL_REGULAR_GRID || f->accel == RTB_ACCEL_FLAT_GRID) && f->grid_words)
        t += r((double)f->n_cellwords, 8) + r((double)f->n_cells_used + 1, 4) + r((double)f->n_cell_refs, 4);
    if ((f->accel == RTB_ACCEL_KD_MEDIAN || f->accel == RTB_ACCEL_KD_SAH) && f->kd_nodes) t += r(f->n_kd_nodes, 8) + r((double)f->n_kd_refs, 4);
    if (f->accel == RTB_ACCEL_CONVEX || f->accel == RTB_ACCEL_CONVEX_SIMPLE)
    {
        const double cells = (double)f->cx_table_size * f->cx_table_size;
        t += r(f->n_cx_path, 32) + r(f->n_cx_edges, 12) + r(cells, 1) + r(cells, 4) + r(72000.0 * f->n_cx_edges, 2);
    }
    return t + 4096;
}

// Temporaries of the per-record hierarchy builds and refits, sized for the largest record; released stream-ordered.
struct MeshScratch
{
    cudaStream_t st = nullptr;
    size_t maxN = 0, tmpBytes = 0;
    unsigned int *bounds = nullptr, *arrivals = nullptr;
    unsigned long long *keys = nullptr, *sorted = nullptr;
    int *parent = nullptr; // inner nodes' links at [0, maxN), leaves' at [maxN, 2 maxN)
    void *tmp = nullptr;
    std::vector<void *> temps;
    // rebuild = false: only what a refit or the moments use (arrivals and parent links)
    cudaError_t alloc(cudaStream_t stream, size_t n, bool rebuild)
    {
        st = stream;
        maxN = n;
        auto temp = [&](size_t bytes, void **p) { cudaError_t e = cudaMallocAsync(p, bytes ? bytes : 1, st); if (e == cudaSuccess) temps.push_back(*p); return e; };
        cudaError_t e;
        if ((e = temp(maxN * sizeof(unsigned int), (void **)&arrivals)) != cudaSuccess) return e;
        if ((e = temp(2 * maxN * sizeof(int), (void **)&parent)) != cudaSuccess) return e;
        if (!rebuild) return cudaSuccess;
        if ((e = cub::DeviceRadixSort::SortKeys(nullptr, tmpBytes, keys, sorted, (int)maxN, 0, 62, st)) != cudaSuccess) return e;
        if ((e = temp(6 * sizeof(unsigned int), (void **)&bounds)) != cudaSuccess) return e;
        if ((e = temp(maxN * sizeof(unsigned long long), (void **)&keys)) != cudaSuccess) return e;
        if ((e = temp(maxN * sizeof(unsigned long long), (void **)&sorted)) != cudaSuccess) return e;
        return temp(tmpBytes, &tmp);
    }
    ~MeshScratch() { for (void *p : temps) cudaFreeAsync(p, st); }
};

// The moments of MESH record i (k_bvh_moments) into `moments` (the scene's array, 4 float4 per node slot) from its leaf-order
// records and its tree; the parent links in `t` must be the tree's (k_bvh_hierarchy or k_bvh_parents wrote them).  Uses the
// arrival counters of `t` and allocates nothing.
static int meshMoments(rtb_ctx *ctx, const rtb_scene *s, int i, MeshScratch &t, float4 *moments)
{
    const DScene &d = s->d;
    const int n = d.prims[i].count;
    const unsigned int tb = 256, nb = (unsigned int)((n + tb - 1) / tb);
    const size_t base = (size_t)d.mesh_base[i];
    CUDA_TRY(ctx, cudaMemsetAsync(t.arrivals, 0, (size_t)n * sizeof(unsigned int), t.st));
    k_bvh_moments<<<nb, tb, 0, t.st>>>(d.mesh_tris + 3 * base, n, reinterpret_cast<const rtb_bvhnode *>(d.mesh_nodes) + base, t.parent,
                                       t.parent + t.maxN, t.arrivals, reinterpret_cast<float *>(moments + 4 * base));
    CUDA_TRY(ctx, cudaGetLastError());
    return RTB_OK;
}

// The hierarchy of MESH record i from its raw records `raw` ([count][12] on the device) and its packed records, already in
// DScene::loose.  rebuild: the whole LBVH pipeline (what rtb_scene_upload runs); otherwise a refit: child links and leaf
// order are kept, every box is computed again from the new records.  Moments, once the scene has them, follow either way.
static int meshRecord(rtb_ctx *ctx, rtb_scene *s, int i, const float *raw, MeshScratch &t, bool rebuild)
{
    DScene &d = s->d;
    const cudaStream_t st = t.st;
    const rtb_prim &P = d.prims[i];
    const int n = P.count;
    const unsigned int tb = 256, nb = (unsigned int)((n + tb - 1) / tb), nbInner = (unsigned int)((n - 1 + tb - 1) / tb);
    const size_t base = (size_t)d.mesh_base[i];
    rtb_bvhnode *nodes = reinterpret_cast<rtb_bvhnode *>(const_cast<float4 *>(d.mesh_nodes)) + base;
    uint32_t *order = const_cast<uint32_t *>(d.mesh_order) + base;
    if (rebuild)
    {
        CUDA_TRY(ctx, cudaMemsetAsync(t.bounds, 0xff, 3 * sizeof(unsigned int), st));
        CUDA_TRY(ctx, cudaMemsetAsync(t.bounds + 3, 0, 3 * sizeof(unsigned int), st));
        k_bvh_bounds<<<nb, tb, 0, st>>>(raw, n, t.bounds);
        k_bvh_keys<<<nb, tb, 0, st>>>(raw, n, t.bounds, t.keys);
        size_t need = t.tmpBytes;
        CUDA_TRY(ctx, cub::DeviceRadixSort::SortKeys(t.tmp, need, t.keys, t.sorted, n, 0, 62, st));
        if (n > 1) k_bvh_hierarchy<<<nbInner, tb, 0, st>>>(t.sorted, n, nodes, t.parent, t.parent + t.maxN);
        k_bvh_order<<<nb, tb, 0, st>>>(t.sorted, n, order);
    }
    else if (n > 1) k_bvh_parents<<<nbInner, tb, 0, st>>>(nodes, n, t.parent, t.parent + t.maxN);
    CUDA_TRY(ctx, cudaMemsetAsync(t.arrivals, 0, (size_t)n * sizeof(unsigned int), st));
    k_bvh_boxes<<<nb, tb, 0, st>>>(raw, order, n, nodes, t.parent, t.parent + t.maxN, t.arrivals);
    k_bvh_leaves<<<nb, tb, 0, st>>>(d.loose + 3ull * (unsigned int)P.first, order, n, const_cast<float4 *>(d.mesh_tris) + 3 * base);
    CUDA_TRY(ctx, cudaGetLastError());
    return s->mesh_moments ? meshMoments(ctx, s, i, t, const_cast<float4 *>(s->mesh_moments)) : RTB_OK;
}

// Hierarchies of the MESH records (rtb_build_bvh.cuh) from the raw loose records on the device.  Every record gets its own
// slice of the three arrays (DScene::mesh_base: the mesh triangles of the records before it), so records whose loose ranges
// overlap each have their own tree; a mesh of n triangles uses max(n - 1, 1) <= n node slots (the spare one stays zero).
static int buildMeshesOnDevice(rtb_ctx *ctx, rtb_scene *s, const float *d_raw)
{
    DScene &d = s->d;
    cudaStream_t st = ctx->stream;
    int rc;
    size_t total = 0, maxN = 0;
    for (int i : s->mesh_prims)
    {
        d.mesh_base[i] = (int)total;
        total += (size_t)d.prims[i].count;
        maxN = std::max(maxN, (size_t)d.prims[i].count);
    }
    if (total > 0x7fffffffull) return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scene_upload: more than 2^31 - 1 mesh triangles in all");
    rtb_bvhnode *nodes = nullptr;
    float4 *tris = nullptr;
    uint32_t *order = nullptr;
    if ((rc = deviceArray(ctx, s, total, &nodes, true)) != RTB_OK) return rc;
    if ((rc = deviceArray(ctx, s, 3 * total, &tris, true)) != RTB_OK) return rc;
    if ((rc = deviceArray(ctx, s, total, &order, true)) != RTB_OK) return rc;
    CUDA_TRY(ctx, cudaMemsetAsync(nodes, 0, total * sizeof(rtb_bvhnode), st));
    d.mesh_nodes = reinterpret_cast<const float4 *>(nodes);
    d.mesh_tris = tris;
    d.mesh_order = order;
    MeshScratch t;
    CUDA_TRY(ctx, t.alloc(st, maxN, true));
    for (int i : s->mesh_prims)
        if ((rc = meshRecord(ctx, s, i, d_raw + 12ull * (unsigned int)d.prims[i].first, t, true)) != RTB_OK) return rc;
    return RTB_OK;
}

static int sceneUpload(rtb_ctx *ctx, const rtb_flat_scene *f, rtb_scene **out, bool validate);

extern "C" int rtb_scene_upload(rtb_ctx *ctx, const rtb_flat_scene *f, rtb_scene **out) { return sceneUpload(ctx, f, out, true); }

// validate = false skips the whole-stream index / structure checks: only for a flat scene that has just passed them on another
// device of the same rtb_multi (the cheap header checks always run)
static int sceneUpload(rtb_ctx *ctx, const rtb_flat_scene *f, rtb_scene **out, bool validate)
{
    UploadLaps laps;
    if (!ctx || !f || !out) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: null argument");
    *out = nullptr;
    if (f->n_prims <= 0 || !f->prims) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: empty scene");
    if (f->n_prims > RTB_MAX_INLINE_PRIMS)
        return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scene_upload: more than 16 top-level records (runs of loose triangles count once)");
    if (f->n_materials <= 0 || f->n_materials > RTB_MAX_INLINE_MATS || !f->materials)
        return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scene_upload: between 1 and 16 materials are supported");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));

    rtb_scene *s = new rtb_scene();
    DScene &d = s->d;
    memset(&d, 0, sizeof(d));
    if (cudaEventCreateWithFlags(&s->last_use, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ready, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->query_use, cudaEventDisableTiming) != cudaSuccess)
    {
        rtb_scene_free(ctx, s);
        return fail(ctx, RTB_ERR_CUDA, "rtb_scene_upload: cudaEventCreate failed");
    }
    d.n_prims = f->n_prims; d.n_materials = f->n_materials; d.n_top = f->n_top; d.accel = f->accel;
    int tunnels = 0;
    for (int i = 0; i < f->n_prims; i++)
    {
        const rtb_prim &p = f->prims[i];
        d.prims[i] = p;
        bool ok = p.type >= RTB_PRIM_PLANE && p.type <= RTB_PRIM_MESH;
        if (p.type != RTB_PRIM_TUNNEL) ok = ok && p.material >= 0 && p.material < f->n_materials;
        if (p.type == RTB_PRIM_TRIANGLES || p.type == RTB_PRIM_MESH)
            ok = ok && p.first >= 0 && p.count >= 0 && (int64_t)p.first + p.count <= f->n_loose && f->loose_tri;
        if (p.type == RTB_PRIM_MESH) { ok = ok && p.count >= 1; s->mesh_prims.push_back(i); }
        if (p.type == RTB_PRIM_TUNNEL) tunnels++;
        if (!ok) { rtb_scene_free(ctx, s); return fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: bad top-level record " + std::to_string(i)); }
    }
    if (tunnels > 1) { rtb_scene_free(ctx, s); return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scene_upload: one tunnel per scene"); }
    s->has_tunnel = tunnels == 1;
    s->has_mesh = !s->mesh_prims.empty();
    for (int i = 0; i < f->n_materials; i++)
    {
        d.mats[i] = f->materials[i];
        if (f->materials[i].refractiveness > 0) s->has_refractive = true;
    }

    int rc = RTB_OK;
    ctx->sources_page_locked = f->arrays_page_locked != 0;
    BackgroundChecks checks;
    checks.enabled = validate;
    auto bail = [&](int code) {
        checks.join();
        if (s->direct_sources) cudaStreamSynchronize(ctx->stream); // queued copies read the caller's arrays
        rtb_scene_free(ctx, s);
        return code;
    };
    // The whole-array checks start first, on the context's checker threads: with page-locked source arrays nothing else of an
    // upload takes as long (SAH scene: 0.45 ms for the tree's shape alone when it was one pass on one thread).
    if (validate && s->has_tunnel)
    {
        if (!ctx->checkers) { ctx->checkers = new WorkerPool(); ctx->checkers->start(8); }
        checks.pool = ctx->checkers;
        queueSceneChecks(f, checks);
        checks.start();
    }
    laps.lap("header + checks queued");

    // every stream is packed / copied into the page-locked staging ring and leaves with an asynchronous copy:
    // no intermediate synchronisation, the upload is ordered before the renders on ctx->stream
    const size_t nLoose = f->loose_tri ? (size_t)f->n_loose : 0;
    {
        float *d_rawLoose = nullptr; // kept for the mesh builds
        if ((rc = uploadTriangles(ctx, s, f->loose_tri, nLoose, &d.loose, nullptr, s->has_mesh ? &d_rawLoose : nullptr)) != RTB_OK) return bail(rc);
        if (s->has_mesh)
        {
            rc = buildMeshesOnDevice(ctx, s, d_rawLoose);
            cudaFreeAsync(d_rawLoose, ctx->stream);
            if (rc != RTB_OK) return bail(rc);
            laps.lap("mesh hierarchies");
        }
    }

    if (s->has_tunnel)
    {
        if (f->n_tris < 0 || (f->n_tris > 0 && (!f->tri || !f->tri_material)))
            return bail(fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: tunnel triangle streams missing"));
        uint32_t maxMat = 0; // negative ids wrap to huge values
        for (int i = 0; validate && i < f->n_tris; i++) maxMat = (uint32_t)f->tri_material[i] > maxMat ? (uint32_t)f->tri_material[i] : maxMat;
        if (f->n_tris > 0 && maxMat >= (uint32_t)f->n_materials)
            return bail(fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: triangle material out of range"));
        const size_t nTris = (size_t)f->n_tris;
        laps.lap("loose+material check");
        const bool gridAccel = f->accel == RTB_ACCEL_REGULAR_GRID || f->accel == RTB_ACCEL_FLAT_GRID;
        const bool gridOnDevice = gridAccel && !f->grid_words && f->grid_build_resolution > 1;
        const bool kdOnDevice = f->accel == RTB_ACCEL_KD_SAH && !f->kd_nodes && f->kd_build_max_depth > 0;
        float *d_raw = nullptr; // kept for a device accelerator build
        if ((rc = uploadTriangles(ctx, s, f->tri, nTris, &d.tri, &d.tri_pre, (gridOnDevice || kdOnDevice) ? &d_raw : nullptr)) != RTB_OK) return bail(rc);
        struct RawGuard { float *&p; cudaStream_t st; ~RawGuard() { if (p) cudaFreeAsync(p, st); } } rawGuard{d_raw, ctx->stream};
        if ((rc = uploadArray(ctx, s, f->tri_material, nTris, &d.tri_material)) != RTB_OK) return bail(rc);
        d.n_tris = f->n_tris;
        laps.lap("triangle streams");

        if (gridOnDevice)
        { // no grid arrays, a resolution: build it here, on the device
            if (f->n_tris <= 0) return bail(fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: a grid needs triangles"));
            if ((rc = buildGridOnDevice(ctx, s, f, d_raw)) != RTB_OK) return bail(rc);
        }
        else if (f->accel == RTB_ACCEL_REGULAR_GRID || f->accel == RTB_ACCEL_FLAT_GRID)
        {
            if (!gridHeaderOk(f)) return bail(fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: inconsistent grid directory"));
            // (the whole-array checks of the directory and the references are running: queueSceneChecks above)
            d.g_origin = {f->grid_origin[0], f->grid_origin[1], f->grid_origin[2]};
            d.g_cell = {f->grid_cell[0], f->grid_cell[1], f->grid_cell[2]};
            d.nx = f->grid_dims[0]; d.ny = f->grid_dims[1]; d.nz = f->grid_dims[2];
            // reference Tunnel.cpp:822-825: far = origin + Vector(cellSize * length)
            d.g_extent = {d.g_cell.x * d.nx, d.g_cell.y * d.ny, d.g_cell.z * d.nz};
            d.g_far = {d.g_origin.x + d.g_extent.x, d.g_origin.y + d.g_extent.y, d.g_origin.z + d.g_extent.z};
            const uint2 *words = nullptr;
            if ((rc = uploadArray(ctx, s, (const uint2 *)f->grid_words, (size_t)f->n_cellwords, &words)) != RTB_OK) return bail(rc);
            d.g_words = words;
            if ((rc = uploadArray(ctx, s, f->grid_cell_start, (size_t)f->n_cells_used + 1, &d.g_start)) != RTB_OK) return bail(rc);
            if ((rc = uploadArray(ctx, s, f->grid_cell_tris, (size_t)f->n_cell_refs, &d.g_tris)) != RTB_OK) return bail(rc);
            // k_pack_pairs indexes the triangle stream with these references: the verdict of the checks comes first
            if ((rc = collectVerdict(ctx, checks)) != RTB_OK) return bail(rc);
            if ((rc = packPairs(ctx, s, d.g_tris, (size_t)f->n_cell_refs)) != RTB_OK) return bail(rc);
            s->grid_cells_used = f->n_cells_used; s->grid_refs = f->n_cell_refs; s->grid_words = f->n_cellwords;
        }
        else if (kdOnDevice)
        { // no node arrays, build parameters: the SAH tree is built here, on the device
            if (f->n_tris <= 0) return bail(fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: a k-d tree needs triangles"));
            if ((rc = buildKdOnDevice(ctx, s, f, d_raw)) != RTB_OK) return bail(rc);
        }
        else if (f->accel == RTB_ACCEL_KD_MEDIAN || f->accel == RTB_ACCEL_KD_SAH)
        {
            if (!kdHeaderOk(f)) return bail(fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: k-d tree missing"));
            d.kd_min = {f->kd_min[0], f->kd_min[1], f->kd_min[2]};
            // reference Grid.cpp:13-17: Grid(near, far) keeps size = far - near
            d.kd_size = {f->kd_max[0] - f->kd_min[0], f->kd_max[1] - f->kd_min[1], f->kd_max[2] - f->kd_min[2]};
            const uint2 *nodes = nullptr;
            if ((rc = uploadArray(ctx, s, (const uint2 *)f->kd_nodes, (size_t)f->n_kd_nodes, &nodes)) != RTB_OK) return bail(rc);
            d.kd_nodes = nodes;
            if ((rc = uploadArray(ctx, s, f->kd_leaf_tris, (size_t)f->n_kd_refs, &d.kd_tris)) != RTB_OK) return bail(rc);
            // k_pack_pairs indexes the triangle stream with these references: the verdict of the checks comes first
            laps.lap("k-d arrays queued");
            if ((rc = collectVerdict(ctx, checks)) != RTB_OK) return bail(rc);
            laps.lap("verdict");
            s->kd_nodes = f->n_kd_nodes; s->kd_refs = f->n_kd_refs;
            if ((rc = padKdLists(ctx, s, validate ? checks.kd_padded.load() : paddedKdRefs(f))) != RTB_OK) return bail(rc);
        }
        else if (f->accel == RTB_ACCEL_CONVEX || f->accel == RTB_ACCEL_CONVEX_SIMPLE)
        {
            const int64_t perSegment = 2 * (int64_t)f->n_cx_edges;
            if (f->n_cx_path < 2 || f->n_cx_edges < 3 || f->n_cx_edges > 32767 || !f->cx_frames || !f->cx_edges || !f->cx_cell_status ||
                !f->cx_cell_range || (f->accel == RTB_ACCEL_CONVEX && !f->cx_order) || !(f->cx_width > 0) || !(f->cx_height > 0) ||
                f->cx_table_size < 2 || f->cx_table_size > 4096)
                return bail(fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: convex accelerator tables missing (the tunnel needs ring normals: "
                                                       "PerformanceTest's generator)"));
            if ((int64_t)f->n_tris != (f->n_cx_path - 1) * perSegment)
                return bail(fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: convex accelerator needs (n_cx_path - 1) * 2 * n_cx_edges triangles in segment order"));
            const size_t tableCells = (size_t)f->cx_table_size * f->cx_table_size;
            for (size_t i = 0; validate && i < tableCells; i++)
            {
                const int st = f->cx_cell_status[i], b = f->cx_cell_range[2 * i], e = f->cx_cell_range[2 * i + 1];
                if (st > 2 || (st == 1 && (b < 0 || e >= f->n_cx_edges)))
                    return bail(fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: bad convex cell table"));
            }
            if (f->accel == RTB_ACCEL_CONVEX && validate)
                for (int64_t i = 0; i < (int64_t)100 * 360 * perSegment; i++)
                    if (f->cx_order[i] >= perSegment) return bail(fail(ctx, RTB_ERR_INVALID, "rtb_scene_upload: bad convex order table"));
            d.cx_n_path = f->n_cx_path; d.cx_n_edges = f->n_cx_edges; d.cx_width = f->cx_width; d.cx_height = f->cx_height;
            d.cx_table = f->cx_table_size; d.cx_round_bins = f->cx_round_bins ? 1 : 0;
            if ((rc = uploadArray(ctx, s, f->cx_frames, (size_t)f->n_cx_path * 8, &d.cx_frames)) != RTB_OK) return bail(rc);
            if ((rc = uploadArray(ctx, s, f->cx_edges, (size_t)f->n_cx_edges * 3, &d.cx_edges)) != RTB_OK) return bail(rc);
            if ((rc = uploadArray(ctx, s, f->cx_cell_status, tableCells, &d.cx_status)) != RTB_OK) return bail(rc);
            if ((rc = uploadArray(ctx, s, (const short *)f->cx_cell_range, tableCells * 2, &d.cx_range)) != RTB_OK) return bail(rc);
            if (f->accel == RTB_ACCEL_CONVEX &&
                (rc = uploadArray(ctx, s, f->cx_order, (size_t)100 * 360 * perSegment, &d.cx_order)) != RTB_OK) return bail(rc);
        }
        else if (f->accel != RTB_ACCEL_LINEAR)
            return bail(fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scene_upload: unknown accelerator"));
    }
    // no synchronisation: the copies are queued on ctx->stream ahead of anything that reads the scene; launches on
    // another stream (rtb_render_device) wait for this event
    laps.lap("accelerator");
    if ((rc = collectVerdict(ctx, checks)) != RTB_OK) return bail(rc);
    laps.lap("checks joined");
    {
        const cudaError_t e = cudaEventRecord(s->ready, ctx->stream);
        if (e != cudaSuccess) return bail(fail(ctx, RTB_ERR_CUDA, std::string("cudaEventRecord(ready): ") + cudaGetErrorString(e)));
    }
    s->signature = sceneSignature(f);
    laps.lap("signature");
    s->long_lists = s->has_tunnel && f->accel == RTB_ACCEL_REGULAR_GRID && s->grid_cells_used > 0 && s->grid_refs >= 16 * s->grid_cells_used;
    *out = s;
    return RTB_OK;
}

extern "C" int rtb_scene_free(rtb_ctx *ctx, rtb_scene *s)
{
    if (!s) return RTB_OK;
    if (ctx)
    { // stream-ordered release: after the last launch that read the scene (on whichever stream it ran)
        cudaSetDevice(ctx->device);
        // copies straight out of the caller's page-locked arrays: the caller may reuse them once the scene is freed
        if (s->direct_sources && s->ready && cudaEventQuery(s->ready) != cudaSuccess) { cudaGetLastError(); cudaEventSynchronize(s->ready); }
        if (s->last_use) cudaStreamWaitEvent(ctx->stream, s->last_use, 0);
        if (s->query_use) cudaStreamWaitEvent(ctx->stream, s->query_use, 0);
        for (void *p : s->allocs) cudaFreeAsync(p, ctx->stream);
    }
    else
        for (void *p : s->allocs) cudaFree(p);
    if (s->last_use) cudaEventDestroy(s->last_use);
    if (s->ready) cudaEventDestroy(s->ready);
    if (s->query_use) cudaEventDestroy(s->query_use);
    delete s;
    return RTB_OK;
}

extern "C" int64_t rtb_scene_device_bytes(const rtb_scene *s) { return s ? s->bytes : 0; }
extern "C" int64_t rtb_scene_upload_bytes(const rtb_scene *s) { return s ? s->h2d_bytes : 0; }

extern "C" int rtb_scene_grid_hash(rtb_ctx *ctx, const rtb_scene *s, uint64_t *hash, int64_t stats[6])
{
    if (!ctx || !s || !hash) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_grid_hash: null argument");
    const DScene &d = s->d;
    if (!s->has_tunnel || (d.accel != RTB_ACCEL_REGULAR_GRID && d.accel != RTB_ACCEL_FLAT_GRID))
        return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scene_grid_hash: the scene has no grid");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<uint2> words((size_t)s->grid_words);
    std::vector<uint32_t> start((size_t)s->grid_cells_used + 1), tris((size_t)s->grid_refs);
    CUDA_TRY(ctx, cudaMemcpyAsync(words.data(), d.g_words, words.size() * sizeof(uint2), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(start.data(), d.g_start, start.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(tris.data(), d.g_tris, tris.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    auto mix = [](uint64_t &h, uint32_t v) { h = (h ^ v) * 0x100000001b3ull; };
    auto bits = [](float v) { uint32_t u; memcpy(&u, &v, 4); return u; };
    uint64_t x = 0xcbf29ce484222325ull;
    mix(x, 0x47524944u);
    mix(x, (uint32_t)d.nx); mix(x, (uint32_t)d.ny); mix(x, (uint32_t)d.nz);
    mix(x, bits(d.g_origin.x)); mix(x, bits(d.g_origin.y)); mix(x, bits(d.g_origin.z));
    mix(x, bits(d.g_cell.x)); mix(x, bits(d.g_cell.y)); mix(x, bits(d.g_cell.z));
    int64_t longest = 0;
    for (size_t w = 0; w < words.size(); w++)
    {
        uint32_t b = words[w].x, r = words[w].y;
        while (b)
        {
            const int bit = __builtin_ctz(b);
            b &= b - 1;
            if ((size_t)r + 1 >= start.size()) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_grid_hash: inconsistent cell directory");
            const uint32_t first = start[r], last = start[r + 1];
            mix(x, (uint32_t)(w * 32 + bit));
            mix(x, last - first);
            for (uint32_t e = first; e < last; e++) mix(x, tris[e]);
            if ((int64_t)(last - first) > longest) longest = last - first;
            r++;
        }
    }
    *hash = x;
    if (stats) { stats[0] = d.nx; stats[1] = d.ny; stats[2] = d.nz; stats[3] = s->grid_cells_used; stats[4] = s->grid_refs; stats[5] = longest; }
    return RTB_OK;
}

extern "C" int rtb_scene_kd_download(rtb_ctx *ctx, const rtb_scene *s, rtb_kdnode *nodes, int64_t node_cap, uint32_t *leaf_tris,
                                     int64_t ref_cap, int64_t counts[3], float box[6])
{
    if (!ctx || !s) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_kd_download: null argument");
    const DScene &d = s->d;
    if (!s->has_tunnel || (d.accel != RTB_ACCEL_KD_MEDIAN && d.accel != RTB_ACCEL_KD_SAH))
        return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scene_kd_download: the scene has no k-d tree");
    if (counts) { counts[0] = s->kd_nodes; counts[1] = s->kd_refs; counts[2] = s->kd_levels; }
    if (box) { box[0] = d.kd_min.x; box[1] = d.kd_min.y; box[2] = d.kd_min.z; box[3] = d.kd_size.x; box[4] = d.kd_size.y; box[5] = d.kd_size.z; }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (nodes)
    {
        if (node_cap < s->kd_nodes) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_kd_download: node buffer too small");
        CUDA_TRY(ctx, cudaMemcpyAsync(nodes, s->kd_nodes_plain ? s->kd_nodes_plain : d.kd_nodes, (size_t)s->kd_nodes * sizeof(rtb_kdnode), cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (leaf_tris)
    {
        if (ref_cap < s->kd_refs) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_kd_download: reference buffer too small");
        CUDA_TRY(ctx, cudaMemcpyAsync(leaf_tris, s->kd_tris_plain ? s->kd_tris_plain : d.kd_tris, (size_t)s->kd_refs * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return RTB_OK;
}

extern "C" int rtb_scene_mesh_download(rtb_ctx *ctx, const rtb_scene *s, int32_t mesh_index, rtb_bvhnode *nodes, int64_t node_cap,
                                       uint32_t *tri_order, int64_t tri_cap, int64_t counts[3])
{
    if (!ctx || !s) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_mesh_download: null argument");
    if (mesh_index < 0 || mesh_index >= (int32_t)s->mesh_prims.size())
        return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scene_mesh_download: the scene has no such mesh record");
    const rtb_prim &P = s->d.prims[s->mesh_prims[(size_t)mesh_index]];
    const int64_t nNodes = P.count > 1 ? P.count - 1 : 1;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<rtb_bvhnode> all((size_t)nNodes);
    const size_t base = (size_t)s->d.mesh_base[s->mesh_prims[(size_t)mesh_index]];
    CUDA_TRY(ctx, cudaMemcpyAsync(all.data(), s->d.mesh_nodes + 4 * base, (size_t)nNodes * sizeof(rtb_bvhnode),
                                  cudaMemcpyDeviceToHost, ctx->stream));
    if (tri_order)
    {
        if (tri_cap < P.count) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_mesh_download: order buffer too small");
        CUDA_TRY(ctx, cudaMemcpyAsync(tri_order, s->d.mesh_order + base, (size_t)P.count * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (nodes)
    {
        if (node_cap < nNodes) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_mesh_download: node buffer too small");
        memcpy(nodes, all.data(), (size_t)nNodes * sizeof(rtb_bvhnode));
    }
    if (counts)
    { // depth by an explicit walk; a link outside the node array ends the walk as an error
        int64_t depth = 0;
        std::vector<std::pair<int32_t, int64_t>> stack{{0, 0}};
        int64_t visited = 0;
        while (!stack.empty())
        {
            const auto [node, dep] = stack.back();
            stack.pop_back();
            if (++visited > nNodes) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_mesh_download: malformed tree");
            for (int c = 0; c < (P.count > 1 ? 2 : 1); c++)
            {
                const int32_t ch = all[(size_t)node].child[c];
                if (ch < 0) depth = std::max(depth, dep + 1);
                else if (ch < nNodes) stack.push_back({ch, dep + 1});
                else return fail(ctx, RTB_ERR_INVALID, "rtb_scene_mesh_download: malformed tree");
            }
        }
        counts[0] = nNodes; counts[1] = P.count; counts[2] = depth;
    }
    return RTB_OK;
}

// ---- mesh update ------------------------------------------------------------------------------
// The MESH records an update of record `mesh_index` with n records rewrites: that record, then every other MESH record whose
// range intersects its range (which must lie inside it).  Every check of the update is here, before anything is written.
static int meshUpdateRecords(rtb_ctx *ctx, const rtb_scene *s, int32_t mesh_index, int64_t n, int32_t flags, std::vector<int> &recs)
{
    if (flags != RTB_MESH_REBUILD && flags != RTB_MESH_REFIT) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_mesh_update: unknown flags");
    if (mesh_index < 0 || mesh_index >= (int32_t)s->mesh_prims.size())
        return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scene_mesh_update: the scene has no such mesh record");
    const int target = s->mesh_prims[(size_t)mesh_index];
    const rtb_prim &M = s->d.prims[target];
    if (n != M.count) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_mesh_update: n differs from the mesh record's count");
    const int64_t first = M.first, end = (int64_t)M.first + M.count;
    recs.assign(1, target);
    for (int j : s->mesh_prims)
    {
        const rtb_prim &P = s->d.prims[j];
        const int64_t b = P.first, e = (int64_t)P.first + P.count;
        if (j == target || e <= first || b >= end) continue;
        if (b < first || e > end)
            return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scene_mesh_update: mesh record " + std::to_string(j) +
                                                      " overlaps the updated range only in part");
        recs.push_back(j);
    }
    return RTB_OK;
}

// Enqueue the update on ctx->stream behind `caller` and every launch that has read the scene; `caller` waits for it.  `src`
// holds the records of the whole range: device memory of this device, or page-locked host memory (staged) when `host`.
static int meshUpdateEnqueue(rtb_ctx *ctx, rtb_scene *s, const std::vector<int> &recs, const float *src, bool host, int32_t flags,
                             cudaStream_t caller)
{
    DScene &d = s->d;
    const cudaStream_t st = ctx->stream;
    const rtb_prim &M = d.prims[recs[0]];
    const size_t n = (size_t)M.count, bytes = n * 12 * sizeof(float);
    if (caller != st)
    {
        if (!ctx->caller_ready) CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->caller_ready, cudaEventDisableTiming));
        CUDA_TRY(ctx, cudaEventRecord(ctx->caller_ready, caller));
        CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->caller_ready, 0));
    }
    // renders on other streams record last_use behind their kernels, and frames of a context run one after the other
    // (waitLastFrame): the last one covers them all
    CUDA_TRY(ctx, cudaStreamWaitEvent(st, s->last_use, 0));
    CUDA_TRY(ctx, cudaStreamWaitEvent(st, s->query_use, 0)); // queries on any stream (chained: the last one covers them all)
    // every allocation comes before the first write to the scene: a failed one leaves the scene as it was
    struct RawGuard { void *p = nullptr; cudaStream_t st; ~RawGuard() { if (p) cudaFreeAsync(p, st); } } raw{nullptr, st};
    MeshScratch t;
    if (host) CUDA_TRY(ctx, cudaMallocAsync(&raw.p, bytes, st));
    CUDA_TRY(ctx, t.alloc(st, n, flags == RTB_MESH_REBUILD));
    if (host)
    {
        CUDA_TRY(ctx, cudaMemcpyAsync(raw.p, src, bytes, cudaMemcpyHostToDevice, st));
        src = (const float *)raw.p;
    }
    k_pack_triangles<<<(unsigned int)((n + 255) / 256), 256, 0, st>>>(src, (int)n, const_cast<float4 *>(d.loose) + 3ull * (unsigned int)M.first, nullptr);
    CUDA_TRY(ctx, cudaGetLastError());
    for (int i : recs)
    {
        const int rc = meshRecord(ctx, s, i, src + 12ull * (unsigned int)(d.prims[i].first - M.first), t, flags == RTB_MESH_REBUILD);
        if (rc != RTB_OK) return rc;
    }
    CUDA_TRY(ctx, cudaEventRecord(s->ready, st));
    if (caller != st) CUDA_TRY(ctx, cudaStreamWaitEvent(caller, s->ready, 0));
    return RTB_OK;
}

extern "C" int rtb_scene_mesh_update(rtb_ctx *ctx, rtb_scene *s, int32_t mesh_index, const float *tri, int64_t n, int32_t flags,
                                     void *stream)
{
    if (!ctx || !s || !tri) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_mesh_update: null argument");
    std::vector<int> recs;
    int rc = meshUpdateRecords(ctx, s, mesh_index, n, flags, recs);
    if (rc != RTB_OK) return rc;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaPointerAttributes attr;
    const bool known = cudaPointerGetAttributes(&attr, tri) == cudaSuccess;
    cudaGetLastError();
    // managed memory may still be written by work on `stream`: it is read on the device, in stream order, like device memory
    const bool managed = known && attr.type == cudaMemoryTypeManaged;
    const bool onDevice = managed || (known && attr.type == cudaMemoryTypeDevice);
    const float *src = tri;
    if (onDevice)
    {
        if (!managed && attr.device != ctx->device) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_mesh_update: the records are on another device");
        if ((uintptr_t)tri & 15u) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_mesh_update: device records must be 16-byte aligned");
    }
    else
    { // staged: the caller may reuse its array when the call returns
        char *staged = nullptr;
        const size_t bytes = (size_t)n * 12 * sizeof(float);
        if ((rc = stageReserve(ctx, bytes, &staged)) != RTB_OK) return rc;
        memcpy(staged, tri, bytes);
        src = (const float *)staged;
    }
    return meshUpdateEnqueue(ctx, s, recs, src, !onDevice, flags, stream ? (cudaStream_t)stream : ctx->stream);
}

extern "C" int rtb_scene_mesh_moments(rtb_ctx *ctx, rtb_scene *s, void *stream)
{
    if (!ctx || !s) return fail(ctx, RTB_ERR_INVALID, "rtb_scene_mesh_moments: null argument");
    if (s->mesh_moments || s->mesh_prims.empty()) return RTB_OK; // built already, or nothing to build
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const DScene &d = s->d;
    const cudaStream_t st = ctx->stream, caller = stream ? (cudaStream_t)stream : st;
    size_t slots = 0, maxN = 0;
    for (int i : s->mesh_prims)
    {
        slots += (size_t)d.prims[i].count;
        maxN = std::max(maxN, (size_t)d.prims[i].count);
    }
    // ordered as a mesh update: behind the caller's stream and every launch that has read the scene
    if (caller != st)
    {
        if (!ctx->caller_ready) CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->caller_ready, cudaEventDisableTiming));
        CUDA_TRY(ctx, cudaEventRecord(ctx->caller_ready, caller));
        CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->caller_ready, 0));
    }
    CUDA_TRY(ctx, cudaStreamWaitEvent(st, s->last_use, 0));
    CUDA_TRY(ctx, cudaStreamWaitEvent(st, s->query_use, 0));
    MeshScratch t;
    CUDA_TRY(ctx, t.alloc(st, maxN, false));
    float4 *moments = nullptr;
    int rc = deviceArray(ctx, s, 4 * slots, &moments, true);
    if (rc != RTB_OK) return rc;
    // the scene has moments only once every launch is enqueued: a failed call releases the array and leaves the scene without
    // them, so a query stays refused and a later call builds them again
    auto failed = [&](int code) {
        s->allocs.pop_back();
        s->bytes -= (int64_t)(4 * slots * sizeof(float4));
        cudaFreeAsync(moments, st);
        return code;
    };
    cudaError_t e = cudaMemsetAsync(moments, 0, 4 * slots * sizeof(float4), st);
    if (e != cudaSuccess) return failed(fail(ctx, RTB_ERR_CUDA, std::string("rtb_scene_mesh_moments: ") + cudaGetErrorString(e)));
    for (int i : s->mesh_prims)
    {
        const int n = d.prims[i].count;
        if (n > 1)
            k_bvh_parents<<<(unsigned int)((n - 1 + 255) / 256), 256, 0, st>>>(reinterpret_cast<const rtb_bvhnode *>(d.mesh_nodes) + d.mesh_base[i],
                                                                              n, t.parent, t.parent + t.maxN);
        if ((rc = meshMoments(ctx, s, i, t, moments)) != RTB_OK) return failed(rc);
    }
    if ((e = cudaEventRecord(s->ready, st)) != cudaSuccess ||
        (caller != st && (e = cudaStreamWaitEvent(caller, s->ready, 0)) != cudaSuccess))
        return failed(fail(ctx, RTB_ERR_CUDA, std::string("rtb_scene_mesh_moments: ") + cudaGetErrorString(e)));
    s->mesh_moments = moments;
    return RTB_OK;
}

// ---- render -----------------------------------------------------------------------------------
static int makeFrame(rtb_ctx *ctx, const rtb_scene *scene, const rtb_camera *cam, const rtb_render_setting *setting,
                     const rtb_frame *frame, FrameParams &F)
{
    if (!ctx || !scene || !cam || !setting || !frame) return fail(ctx, RTB_ERR_INVALID, "render: null argument");
    if (frame->width <= 0 || frame->height <= 0) return fail(ctx, RTB_ERR_INVALID, "render: bad image size");
    const int world = frame->world > 0 ? frame->world : 1;
    if (frame->layout & ~(RTB_LAYOUT_REFERENCE | RTB_LAYOUT_GLOBAL | RTB_OUTPUT_RGB8 | RTB_OUTPUT_MOMENTS))
        return fail(ctx, RTB_ERR_INVALID, "render: unknown layout flags");
    const bool global = (frame->layout & RTB_LAYOUT_GLOBAL) != 0;
    const bool reference = (frame->layout & RTB_LAYOUT_REFERENCE) != 0;
    int64_t rows;
    if (reference && global && colSharded(frame))
    { // the reference order addresses by frame coordinates, so a column-block shard can store into the whole frame too
        rtb_frame plain = *frame;
        plain.layout &= ~RTB_LAYOUT_REFERENCE;
        rows = rtb_shard_rows(&plain);
    }
    else rows = rtb_shard_rows(frame);
    if (rows < 0)
        return fail(ctx, RTB_ERR_INVALID, "render: bad shard (rank / world / row_block: row_block must be a multiple of 8; col_block: a multiple "
                                          "of 8 with width a multiple of world * col_block, row-major layout)");
    if (reference && world != 1 && !global)
        return fail(ctx, RTB_ERR_INVALID, "render: the reference (column-major) layout needs the whole frame in one buffer (one rank, or RTB_LAYOUT_GLOBAL)");
    const bool moments = (frame->layout & RTB_OUTPUT_MOMENTS) != 0;
    if (moments && (!setting->enable_monte_carlo || reference || (frame->layout & RTB_OUTPUT_RGB8)))
        return fail(ctx, RTB_ERR_INVALID, "render: RTB_OUTPUT_MOMENTS needs a Monte-Carlo setting and a row-major float buffer");
    int sFirst = 0, sEnd = frame->samples;
    if (setting->enable_monte_carlo)
    {
        if (frame->samples <= 0) return fail(ctx, RTB_ERR_INVALID, "render: samples must be positive");
        if (frame->sample_count != 0 || frame->sample_first != 0)
        {
            if (frame->sample_first < 0 || frame->sample_count <= 0 || (int64_t)frame->sample_first + frame->sample_count > frame->samples)
                return fail(ctx, RTB_ERR_INVALID, "render: sample shard outside [0, samples)");
            sFirst = frame->sample_first; sEnd = sFirst + frame->sample_count;
        }
        int need = setting->single_tracing_depth;
        if (setting->max_depth < need) need = setting->max_depth;
        if (need > RTB_MAX_DEPTH) need = RTB_MAX_DEPTH;
        if (need > RTB_MC_STACK)
            return fail(ctx, RTB_ERR_UNSUPPORTED, "render: min(single_tracing_depth, max_depth) above 32 pending split rays");
    }
    else if (scene->has_refractive && setting->max_depth > (RTB_TREE_STACK - 3) / 2)
        return fail(ctx, RTB_ERR_UNSUPPORTED, "render: Whitted with refractive materials supports max_depth <= 30");
    memset(&F, 0, sizeof(F));
    F.cam = *cam;
    F.setting = *setting;
    F.width = frame->width; F.height = frame->height; F.samples = frame->samples;
    F.sample_first = sFirst; F.sample_end = sEnd;
    F.rank = frame->rank; F.world = world; F.row_block = normRowBlock(frame);
    F.layout = frame->layout & RTB_LAYOUT_REFERENCE;
    F.rgb8 = (frame->layout & RTB_OUTPUT_RGB8) ? 1 : 0;
    F.moments = moments ? 1 : 0;
    F.global_out = (global && !reference) ? 1 : 0; // the reference order is addressed by frame coordinates anyway
    F.n_local_rows = (int)rows;
    F.col_block = colSharded(frame) ? frame->col_block : 0;
    F.local_width = F.col_block ? frame->width / world : frame->width;
    F.tiles_x = (F.local_width + RTB_TILE_W - 1) / RTB_TILE_W;
    F.n_tiles = F.tiles_x * (int)((rows + RTB_TILE_H - 1) / RTB_TILE_H);
    F.cost_map = frame->counters == 2;
    F.warps_per_cta = RTB_CTA_THREADS / 32;
    F.seed = frame->seed;
    return RTB_OK;
}

// bytes of the output buffer a frame's shard stores into when it is NOT the whole frame
static size_t shardBytes(const FrameParams &F)
{
    return (size_t)F.n_local_rows * F.local_width * 3 * (F.rgb8 ? 1 : sizeof(float)) * (F.moments ? 2 : 1);
}
static size_t frameBytes(const FrameParams &F)
{
    return (size_t)F.height * F.width * 3 * (F.rgb8 ? 1 : sizeof(float)) * (F.moments ? 2 : 1);
}

static int launchRender(rtb_ctx *ctx, const rtb_scene *scene, FrameParams &F, bool count, float *out, Counters *counters, cudaStream_t stream,
                        int &n_kernels)
{
    n_kernels = 1;
    const int warpsPerCta = RTB_CTA_THREADS / 32;
    const dim3 grid((unsigned int)((F.n_tiles + warpsPerCta - 1) / warpsPerCta));
    static const bool resumable = !(getenv("RTB_CHAIN_SM") && atoi(getenv("RTB_CHAIN_SM")) == 0); // A/B switch for profiling
    const int accel = scene->d.accel;
    const bool grid_accel = accel == RTB_ACCEL_REGULAR_GRID || accel == RTB_ACCEL_FLAT_GRID;
    const bool kd_accel = accel == RTB_ACCEL_KD_MEDIAN || accel == RTB_ACCEL_KD_SAH;
    F.skip_heavy = 0;
    F.record_cost = 1;
    auto L = [&](const FrameParams &P, dim3 g, cudaStream_t st) { Launch l; l.S = &scene->d; l.F = &P; l.out = out; l.counters = counters; l.grid = g; l.stream = st; l.count = count; l.mesh = scene->has_mesh; return l; };
    if (F.setting.enable_monte_carlo) launchMonteCarlo(L(F, grid, stream));
    else if (scene->has_refractive) launchTree(L(F, grid, stream));
    else if (scene->has_mesh) launchChain(L(F, grid, stream)); // the latency tiers have no mesh walk
    else if (resumable && scene->has_tunnel && (kd_accel || grid_accel) && F.order && ctx->tiers_ok)
    { // A tile order is known.  Three kernels share the frame, all launched at once:
      //   order[0 .. n_wide)         the very heaviest tiles: one warp per pixel        (side stream, high priority)
      //   order[n_wide .. n_heavy)   latency-critical tiles: resumable per-lane walk    (side stream, high priority)
      //   order[n_heavy .. n_tiles)  everything else: per-ray walk                      (caller's stream)
      // The regular grid renders ALL remaining tiles with the resumable walk (1.75x faster than per-ray there).
        const bool smallShard = F.n_tiles <= splitMaxTiles();
        const int heavyCap = heavyLimit(F.n_tiles) + wideCount(F.n_tiles, scene->long_lists); // upper bound of the device-side count
        CUDA_TRY(ctx, cudaEventRecord(ctx->fork, stream));
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->aux, ctx->fork, 0));
        const int nWide = wideCount(F.n_tiles, scene->long_lists);
        F.n_wide = (unsigned int)nWide;
        F.heavy_cap = (unsigned int)heavyCap;
        if (nWide > 0)
        {
            FrameParams Wd = F;
            Wd.record_cost = 0;
            Wd.warps_per_cta = warpsPerCta;
            const dim3 wgrid(((unsigned int)nWide * 32u + warpsPerCta - 1) / warpsPerCta);
            launchChainWide(L(Wd, wgrid, ctx->aux));
            n_kernels++;
        }
        // k_whitted_chain_oct is the latency tier of small k-d shards: worst 1/8 shard of the 4K frame SAH 1.99 -> 1.42 ms,
        // k-d median 4.48 -> 3.41, 1280x960 SAH 1.78 -> 1.44 (gpurun_out/sweep5.log, sweep6.log).  Not for a whole 4K
        // frame (throughput-bound: 6.01 -> 6.85 ms) and not for the grids (flat grid 3.20 -> 3.30, regular grid: no gain
        // next to the warp-per-pixel tier, sweep7.log): those keep the resumable walk.
        static const int octTierForced = (int)tunable("RTB_OCT_TIER", -1);
        const int octTier = octTierForced >= 0 ? octTierForced : (smallShard && kd_accel);
        if (accel == RTB_ACCEL_REGULAR_GRID)
        { // one resumable launch for everything after the wide tiles
            FrameParams H = F;
            H.after_wide = 1;
            launchChainSm(L(H, grid, stream), true); // records: it is this frame's throughput kernel
            CUDA_TRY(ctx, cudaEventRecord(ctx->join, ctx->aux));
            CUDA_TRY(ctx, cudaStreamWaitEvent(stream, ctx->join, 0));
        }
        else
        {
            // Small shards (multi-GPU ranks, small frames) are bound by the latency of the heaviest chains, not by
            // issue slots: there each latency-critical tile is walked by 4 warps of 8 lanes (less per-step waiting
            // inside a warp, 4x the warps in flight).  On a big shard the extra warp-instructions would cost more
            // than the shorter tail saves.
            FrameParams H = F;
            H.skip_heavy = 1;
            H.after_wide = 1;
            H.split4 = smallShard ? 1 : 0;
            H.record_cost = 0;
            if (heavyLimit(F.n_tiles) > 0 && octTier)
            { // eight lanes per pixel, eight warps per tile
                H.skip_heavy = 0; H.after_wide = 0; H.split4 = 0;
                H.item_base = F.n_wide; H.item_end = F.n_wide + (unsigned int)heavyLimit(F.n_tiles);
                const dim3 ogrid(((unsigned int)heavyLimit(F.n_tiles) * (unsigned int)octWarpsPerTile(accel, F.n_tiles) + warpsPerCta - 1) / warpsPerCta);
                launchChainOct(L(H, ogrid, ctx->aux), grid_accel);
                n_kernels++;
            }
            else if (heavyLimit(F.n_tiles) > 0)
            {
                const unsigned int heavyWarps = (unsigned int)heavyLimit(F.n_tiles) * (H.split4 ? 4u : 1u);
                const dim3 sgrid((heavyWarps + warpsPerCta - 1) / warpsPerCta);
                launchChainSm(L(H, sgrid, ctx->aux), grid_accel);
                n_kernels++;
            }
            CUDA_TRY(ctx, cudaEventRecord(ctx->join, ctx->aux));
            F.skip_heavy = 1;
            launchChain(L(F, grid, stream));
            CUDA_TRY(ctx, cudaStreamWaitEvent(stream, ctx->join, 0));
        }
    }
    else if (resumable && scene->has_tunnel && accel == RTB_ACCEL_REGULAR_GRID) launchChainSm(L(F, grid, stream), true);
    else launchChain(L(F, grid, stream));
    return RTB_OK;
}

// The scheduling state of a context (d_cost, d_order, d_heavy, d_hist, d_counters, the side stream) is shared by all
// its frames.  Frames are ordered through `last_frame`, recorded behind each frame's last kernel on whatever stream it
// ran: a frame on another stream, and anything that frees or regrows the state, waits for it first.
static bool groupStoreEnabled()
{
    static const bool on = !(getenv("RTB_GROUP_STORE") && atoi(getenv("RTB_GROUP_STORE")) == 0);
    return on;
}

static int waitLastFrame(rtb_ctx *ctx, cudaStream_t stream)
{
    if (ctx->frame_pending && stream != ctx->last_frame_stream) CUDA_TRY(ctx, cudaStreamWaitEvent(stream, ctx->last_frame, 0));
    return RTB_OK;
}

// Attach the tile order learnt from the previous frame of the same geometry (if any) and the cost buffer
static int prepareTileOrder(rtb_ctx *ctx, const rtb_scene *scene, FrameParams &F)
{
    if ((size_t)F.n_tiles > ctx->tile_capacity)
    {
        if (ctx->frame_pending) CUDA_TRY(ctx, cudaEventSynchronize(ctx->last_frame)); // a frame on a caller's stream may still use the buffers
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        if (ctx->d_cost) CUDA_TRY(ctx, cudaFreeAsync(ctx->d_cost, ctx->stream));
        ctx->d_cost = nullptr;
        if (ctx->d_order) CUDA_TRY(ctx, cudaFreeAsync(ctx->d_order, ctx->stream));
        ctx->d_order = nullptr;
        ctx->tile_capacity = 0;
        ctx->order_valid = false;
        CUDA_TRY(ctx, cudaMallocAsync(&ctx->d_cost, (size_t)F.n_tiles * sizeof(unsigned int), ctx->stream));
        CUDA_TRY(ctx, cudaMallocAsync(&ctx->d_order, (size_t)F.n_tiles * sizeof(unsigned int), ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->tile_capacity = (size_t)F.n_tiles;
    }
    if (!ctx->d_hist)
    {
        CUDA_TRY(ctx, cudaMalloc(&ctx->d_hist, RTB_COST_BUCKETS * sizeof(unsigned int)));
        CUDA_TRY(ctx, cudaMalloc(&ctx->d_cursor, RTB_COST_BUCKETS * sizeof(unsigned int)));
        CUDA_TRY(ctx, cudaMemset(ctx->d_hist, 0, RTB_COST_BUCKETS * sizeof(unsigned int)));
        CUDA_TRY(ctx, cudaMalloc(&ctx->d_heavy, 2 * sizeof(unsigned int))); // [0] latency-critical tiles, [1] floor bucket
        CUDA_TRY(ctx, cudaMemset(ctx->d_heavy, 0, 2 * sizeof(unsigned int)));
    }
    // The order (and the per-tile costs behind it) belongs to one view of one scene: frame geometry, scene,
    // camera and depth setting.  A camera move keeps the order for one frame without the tiers (below); anything
    // else starts over with a raster-order frame that measures every tile.
    OrderKey key;
    memset(&key, 0, sizeof(key));
    key.v[0] = F.width; key.v[1] = F.height; key.v[2] = F.rank; key.v[3] = F.world; key.v[4] = F.row_block; key.v[5] = F.layout | ((long long)F.col_block << 8) | ((long long)F.group4 << 40);
    key.v[6] = F.setting.enable_monte_carlo; key.v[7] = F.n_tiles; key.v[8] = F.setting.max_depth;
    key.v[9] = (long long)F.samples | ((long long)F.sample_first << 20) | ((long long)F.sample_end << 40);
    key.scene_signature = scene->signature;
    key.cam = F.cam;
    ctx->tiers_ok = true;
    if (memcmp(&key, &ctx->order_key, sizeof(key)) != 0)
    {
        OrderKey sameView = key;
        sameView.cam = ctx->order_key.cam;
        if (memcmp(&sameView, &ctx->order_key, sizeof(key)) == 0)
            ctx->tiers_ok = false; // only the camera moved: the last order is still a good guess (temporal coherence), but
                                   // every tile is rendered and re-measured by the throughput kernel this frame
        else
            ctx->order_valid = false;
        memcpy(&ctx->order_key, &key, sizeof(key));
    }
    F.order = ctx->order_valid ? ctx->d_order : nullptr;
    F.cost = ctx->d_cost;
    F.n_heavy = ctx->d_heavy;
    return RTB_OK;
}

extern "C" int rtb_forget_schedule(rtb_ctx *ctx)
{
    if (!ctx) return fail(nullptr, RTB_ERR_INVALID, "rtb_forget_schedule: null context");
    ctx->order_valid = false;
    memset(&ctx->order_key, 0, sizeof(ctx->order_key));
    return RTB_OK;
}

// A frame in flight: what renderFinish needs to collect the statistics once the stream has drained
struct PendingFrame
{
    bool active = false, timed = false;
    cudaStream_t stream = nullptr;
    int n_kernels = 0, n_local_rows = 0, n_tiles = 0;
};

// Queue one frame on `stream`: counters reset, render kernel(s), tile-order kernels, optional copy to h_out.  Nothing
// here waits for the device.  `timed`: bracket the frame with the context's timing events (one timed frame per context
// at a time: rtb_render / stats callers, which finish the frame before they return).
static int renderLaunch(rtb_ctx *ctx, const rtb_scene *scene, FrameParams &F, const rtb_frame *frame, float *d_out,
                        cudaStream_t stream, bool timed, float *h_out, bool host_frame, PendingFrame &P)
{
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    P = PendingFrame();
    P.stream = stream;
    P.n_local_rows = F.n_local_rows;
    if (F.n_local_rows == 0) return RTB_OK;
    if (stream != ctx->stream) CUDA_TRY(ctx, cudaStreamWaitEvent(stream, scene->ready, 0)); // the upload ran on ctx->stream
    int rc = waitLastFrame(ctx, stream);
    if (rc != RTB_OK) return rc;
    // whole-tile 128-bit stores (storeTile): row-major frames whose 8-pixel row segments are 16-byte aligned
    static const bool wideStore = !(getenv("RTB_WIDE_STORE") && atoi(getenv("RTB_WIDE_STORE")) == 0);
    F.wide_store = wideStore && !F.layout && !F.cost_map && !F.moments && (F.global_out ? F.width : F.local_width) % 4 == 0 && ((uintptr_t)d_out & 15u) == 0;
    // frames in page-locked host memory: groups of four adjacent tiles per CTA, stored as 384-byte row segments (storeGroup);
    // RTB_GROUP_STORE=0: tile-granular order with the light tiles in raster order, as before
    const bool groupStore = groupStoreEnabled();
    // ... and column-block shards that store into a whole frame in DEVICE memory (RTB_LAYOUT_GLOBAL, 5 ranks and more in bench.py):
    // for all ranks but the owner that frame is peer memory and the stores cross NVLink.  8 B200, 4K SAH step 1.282 -> 1.258 ms;
    // row shards (2 ranks) lose instead, 2.87 -> 2.95 ms: the four tiles of a CTA wait for the slowest one, which costs more than
    // the NVLink writes gain when a rank holds half a frame (profiles/r02_group_store.log).  RTB_GROUP_STORE_PEER=0: off.
    static const bool groupPeer = !(getenv("RTB_GROUP_STORE_PEER") && atoi(getenv("RTB_GROUP_STORE_PEER")) == 0);
    const bool peer_frame = groupPeer && !host_frame && F.global_out && F.world > 1 && F.col_block > 0;
    F.group4 = groupStore && (host_frame || peer_frame) && F.wide_store && !F.setting.enable_monte_carlo && F.tiles_x % 4 == 0 && F.n_local_rows % RTB_TILE_H == 0 &&
               F.local_width % (4 * RTB_TILE_W) == 0 && (!F.col_block || F.col_block % (4 * RTB_TILE_W) == 0);
    // the reference's column-major order (what the RenderProc drop-in asks for), whole frame on this device: blocks of 8x16 pixels
    if (groupStore && host_frame && F.layout == RTB_LAYOUT_REFERENCE && F.world == 1 && !F.cost_map && !F.moments && !F.setting.enable_monte_carlo &&
        F.width % RTB_TILE_W == 0 && F.height % (4 * RTB_TILE_H) == 0 && F.n_local_rows == F.height && ((uintptr_t)d_out & 15u) == 0)
        F.group4 = 2;
    rc = prepareTileOrder(ctx, scene, F); // (the order is keyed by group4 too)
    if (rc != RTB_OK) return rc;
    if (timed) CUDA_TRY(ctx, cudaEventRecord(ctx->ev[0], stream));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_counters, 0, sizeof(Counters), stream));
    if (timed) CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], stream));
    CUDA_TRY(ctx, cudaPeekAtLastError()); // anything stale is reported here, not blamed on the launch
    int n_kernels = 1;
    rc = launchRender(ctx, scene, F, frame->counters != 0, d_out, ctx->d_counters, stream, n_kernels);
    if (rc != RTB_OK) return rc;
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaEventRecord(scene->last_use, stream));
    if (timed) CUDA_TRY(ctx, cudaEventRecord(ctx->ev[2], stream));
    { // heaviest-first order for the next frame of this geometry: counting sort of the recorded tile costs
        int blocks = (F.n_tiles + 1023) / 1024;
        if (blocks > 296) blocks = 296;
        // frames stored straight into host memory order their light tiles by position (k_cost_offsets)
        static const int floorDeltaHost = (int)tunable("RTB_FLOOR_DELTA_HOST", 9), floorDeltaDevice = (int)tunable("RTB_FLOOR_DELTA_DEVICE", 0);
        // Group mode keeps the light tiles in raster order as well -- not for the PCIe write pattern (384-byte segments reach the
        // link's peak in any order) but for an even OUTPUT RATE: in pure heaviest-first order the cheap floor tiles, most of the
        // frame's pixels, all come at the end and the link becomes the bound there (4K SAH frame into host memory, kernel ms at
        // floor 0 / 3 / 6 / 9 / 12 / 16: 5.20 / 5.05 / 4.92 / 4.85 / 4.87 / 4.92; tile-granular stores: 5.11; into HBM: 4.70.
        // A low-discrepancy instead of raster order of the light groups: 4.80-4.85 on SAH, slower on the k-d median tree and
        // the flat grid -- not kept.  profiles/r02_group_store.log)
        static const int floorDeltaGroup = (int)tunable("RTB_FLOOR_DELTA_GROUP", 9);
        // Monte-Carlo frames leave a few bytes per millisecond: pure heaviest-first order for them wherever the frame lies (smallpt
        // 1280x960x64 into host memory, kernel ms with / without the raster-order floor: 40.6 / 37.5 = the device-frame time)
        const int floorDelta = (host_frame && !F.setting.enable_monte_carlo) ? (F.group4 ? floorDeltaGroup : floorDeltaHost) : floorDeltaDevice;
        const int units = F.group4 ? F.n_tiles / 4 : F.n_tiles;
        k_cost_histogram<<<blocks, 256, 0, stream>>>(ctx->d_cost, units, ctx->d_hist, F.group4, F.tiles_x);
        const bool smallShard = F.n_tiles <= splitMaxTiles();
        k_cost_offsets<<<1, RTB_COST_BUCKETS, 0, stream>>>(ctx->d_hist, ctx->d_cursor, ctx->d_heavy, F.n_tiles,
                                             smallShard ? heavyBucketsSmall(scene->d.accel) : RTB_HEAVY_BUCKETS,
                                             heavyLimit(F.n_tiles), wideCount(F.n_tiles, scene->long_lists), floorDelta,
                                             smallShard ? heavyAlpha() : 0.f, 148 * RTB_CHAIN_MIN_CTAS * (RTB_CTA_THREADS / 32));
        k_cost_scatter<<<blocks, 256, 0, stream>>>(ctx->d_cost, units, ctx->d_cursor, ctx->d_order, ctx->d_heavy, F.group4, F.tiles_x);
        CUDA_TRY(ctx, cudaGetLastError());
        ctx->order_valid = true;
    }
    if (h_out) CUDA_TRY(ctx, cudaMemcpyAsync(h_out, d_out, shardBytes(F), cudaMemcpyDeviceToHost, stream));
    if (timed)
    {
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev[3], stream));
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_counters, ctx->d_counters, sizeof(Counters), cudaMemcpyDeviceToHost, stream));
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->last_frame, stream));
    ctx->frame_pending = true;
    ctx->last_frame_stream = stream;
    P.active = true; P.timed = timed; P.n_kernels = n_kernels; P.n_tiles = F.n_tiles;
    return RTB_OK;
}

extern "C" int rtb_set_progress(rtb_ctx *ctx, rtb_progress_fn fn, void *user)
{
    if (!ctx) return fail(nullptr, RTB_ERR_INVALID, "rtb_set_progress: null context");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (fn && !ctx->poll)
    {
        CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->poll, cudaStreamNonBlocking));
        CUDA_TRY(ctx, cudaHostAlloc((void **)&ctx->h_tiles, sizeof(unsigned long long), cudaHostAllocDefault));
    }
    ctx->progress = fn;
    ctx->progress_user = user;
    return RTB_OK;
}

// While the frames in flight on `ctxs` run: read their finished-tile counters over the side streams and report.
// The render kernels are not touched; the reads are 8-byte copies that overlap them.
static void pollProgress(rtb_ctx *const *ctxs, const PendingFrame *P, int n, rtb_progress_fn fn, void *user)
{
    long long total = 0;
    for (int i = 0; i < n; i++) total += P[i].active ? P[i].n_tiles : 0;
    if (!fn || total == 0) return;
    long long last = -1;
    while (true)
    {
        bool running = false;
        long long done = 0;
        for (int i = 0; i < n; i++)
        {
            if (!P[i].active) continue;
            rtb_ctx *c = ctxs[i];
            cudaSetDevice(c->device);
            if (cudaStreamQuery(P[i].stream) == cudaErrorNotReady && c->poll)
            {
                running = true;
                *c->h_tiles = 0;
                if (cudaMemcpyAsync(c->h_tiles, &c->d_counters->tiles, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->poll) == cudaSuccess)
                    cudaStreamSynchronize(c->poll);
                const long long t = (long long)*c->h_tiles;
                done += t < P[i].n_tiles ? t : P[i].n_tiles;
            }
            else done += P[i].n_tiles;
        }
        cudaGetLastError();
        if (!running) break;
        if (done > last) { fn(done, total, user); last = done; }
        std::this_thread::sleep_for(std::chrono::microseconds(250));
    }
    fn(total, total, user);
}

// Wait for a queued frame and collect its statistics (stats may be null)
static int renderFinish(rtb_ctx *ctx, PendingFrame &P, rtb_stats *stats, bool poll = true)
{
    if (stats) memset(stats, 0, sizeof(*stats));
    if (!P.active) return RTB_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (poll && ctx->progress) pollProgress(&ctx, &P, 1, ctx->progress, ctx->progress_user);
    CUDA_TRY(ctx, cudaStreamSynchronize(P.stream));
    if (stats && P.timed)
    {
        const Counters &c = *ctx->h_counters;
        stats->n_rays = (int64_t)c.rays; stats->n_tri_tests = (int64_t)c.tris; stats->n_steps = (int64_t)c.steps;
        stats->n_local_rows = P.n_local_rows;
        CUDA_TRY(ctx, cudaEventElapsedTime(&stats->kernel_ms, ctx->ev[1], ctx->ev[2]));
        CUDA_TRY(ctx, cudaEventElapsedTime(&stats->total_ms, ctx->ev[0], ctx->ev[3]));
        stats->n_launches = P.n_kernels + 3; // render kernel(s) + 3 tile-order kernels
    }
    return RTB_OK;
}

// is `p` page-locked host memory the device can store into?  -> its device alias
static float *hostAlias(void *p)
{
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer) return (float *)attr.devicePointer;
    cudaGetLastError(); // pageable memory: cudaPointerGetAttributes may leave an error behind on older drivers
    return nullptr;
}

extern "C" int rtb_render(rtb_ctx *ctx, const rtb_scene *scene, const rtb_camera *cam, const rtb_render_setting *setting,
                          const rtb_frame *frame, void *rgb_out, rtb_stats *stats)
{
    FrameParams F;
    int rc = makeFrame(ctx, scene, cam, setting, frame, F);
    if (rc != RTB_OK) return rc;
    if (!rgb_out) return fail(ctx, RTB_ERR_INVALID, "rtb_render: null output buffer");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (F.global_out && F.world == 1) F.global_out = 0; // the whole frame on one rank: the same buffer either way
    PendingFrame P;
    { // Page-locked output buffer (rtb_host_alloc / cudaHostAlloc / cudaHostRegister): the kernels store the pixels
      // straight into it over PCIe while they render, instead of a device framebuffer and a copy after the last
      // kernel.  Measured on the 4K SAH frame (scene upload + render + frame in host memory): 9.71 -> 8.77 ms; the
      // kernels slowed down 6.06 -> 7.47 ms under PCIe back-pressure but the 2.4 ms copy was gone; with whole-tile
      // stores and the light tiles in raster order (k_cost_offsets) the slow-down is 5.48 -> 5.75 ms.
        static const bool zerocopy = !(getenv("RTB_ZEROCOPY") && atoi(getenv("RTB_ZEROCOPY")) == 0);
        // 8-bit frames too, provided the tiles leave through storeTile (row-major, width % 4 == 0): 32-bit stores of
        // whole 24-byte row segments with the light tiles in raster order (6.72 -> 6.33 ms); written byte by byte
        // they were slower than a device frame + copy (8.82 vs 7.91 ms)
        static const bool zerocopy8 = !(getenv("RTB_ZEROCOPY_RGB8") && atoi(getenv("RTB_ZEROCOPY_RGB8")) == 0);
        const bool rgb8Direct = zerocopy8 && ((!F.layout && (F.global_out ? F.width : F.local_width) % 4 == 0) ||
                                              (groupStoreEnabled() && F.layout == RTB_LAYOUT_REFERENCE && F.world == 1 && F.width % RTB_TILE_W == 0 && F.height % (4 * RTB_TILE_H) == 0)); // 8x16 blocks
        float *alias = ((zerocopy || F.global_out) && !F.cost_map && (!F.rgb8 || rgb8Direct || F.global_out)) ? hostAlias(rgb_out) : nullptr;
        if (alias)
        {
            rc = renderLaunch(ctx, scene, F, frame, alias, ctx->stream, true, nullptr, true, P);
            if (rc != RTB_OK) return rc;
            return renderFinish(ctx, P, stats);
        }
    }
    if (F.global_out || (F.layout && F.world != 1))
        return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_render: a shard stores into the whole frame (RTB_LAYOUT_GLOBAL) only when the frame is page-locked "
                                              "host memory (rtb_host_alloc); use rtb_render_device for device frames");
    const size_t bytes = shardBytes(F);
    if (bytes > ctx->d_frame_bytes)
    {
        if (ctx->frame_pending) CUDA_TRY(ctx, cudaEventSynchronize(ctx->last_frame));
        if (ctx->d_frame) CUDA_TRY(ctx, cudaFree(ctx->d_frame));
        ctx->d_frame = nullptr;
        ctx->d_frame_bytes = 0;
        CUDA_TRY(ctx, cudaMalloc(&ctx->d_frame, bytes));
        ctx->d_frame_bytes = bytes;
    }
    rc = renderLaunch(ctx, scene, F, frame, ctx->d_frame, ctx->stream, true, (float *)rgb_out, false, P);
    if (rc != RTB_OK) return rc;
    return renderFinish(ctx, P, stats);
}

extern "C" int rtb_render_device(rtb_ctx *ctx, const rtb_scene *scene, const rtb_camera *cam,
                                 const rtb_render_setting *setting, const rtb_frame *frame, void *rgb_device,
                                 void *stream, rtb_stats *stats)
{
    FrameParams F;
    int rc = makeFrame(ctx, scene, cam, setting, frame, F);
    if (rc != RTB_OK) return rc;
    if (!rgb_device) return fail(ctx, RTB_ERR_INVALID, "rtb_render_device: null output buffer");
    PendingFrame P;
    rc = renderLaunch(ctx, scene, F, frame, (float *)rgb_device, stream ? (cudaStream_t)stream : ctx->stream, stats != nullptr, nullptr, false, P);
    if (rc != RTB_OK || !stats) return rc;
    return renderFinish(ctx, P, stats);
}

// ---- one frame buffer, several devices ---------------------------------------------------------------------------
extern "C" int rtb_device_alloc(rtb_ctx *ctx, size_t bytes, void **out)
{
    if (!ctx || !out) return fail(ctx, RTB_ERR_INVALID, "rtb_device_alloc: null argument");
    *out = nullptr;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMalloc(out, bytes ? bytes : 1)); // plain cudaMalloc: pool (cudaMallocAsync) memory cannot be exported
    return RTB_OK;
}

extern "C" int rtb_device_free(rtb_ctx *ctx, void *p)
{
    if (!ctx) return fail(ctx, RTB_ERR_INVALID, "rtb_device_free: null context");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (p) CUDA_TRY(ctx, cudaFree(p));
    return RTB_OK;
}

extern "C" int rtb_device_download(rtb_ctx *ctx, const void *device_ptr, void *host, size_t bytes)
{
    if (!ctx || !device_ptr || !host) return fail(ctx, RTB_ERR_INVALID, "rtb_device_download: null argument");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (ctx->frame_pending) CUDA_TRY(ctx, cudaEventSynchronize(ctx->last_frame));
    CUDA_TRY(ctx, cudaMemcpy(host, device_ptr, bytes, cudaMemcpyDeviceToHost));
    return RTB_OK;
}

static_assert(sizeof(cudaIpcMemHandle_t) == RTB_IPC_HANDLE_BYTES, "RTB_IPC_HANDLE_BYTES must match cudaIpcMemHandle_t");

extern "C" int rtb_ipc_export(rtb_ctx *ctx, void *device_ptr, unsigned char handle[RTB_IPC_HANDLE_BYTES])
{
    if (!ctx || !device_ptr || !handle) return fail(ctx, RTB_ERR_INVALID, "rtb_ipc_export: null argument");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    CUDA_TRY(ctx, cudaIpcGetMemHandle(&h, device_ptr));
    memcpy(handle, &h, sizeof(h));
    return RTB_OK;
}

extern "C" int rtb_ipc_open(rtb_ctx *ctx, const unsigned char handle[RTB_IPC_HANDLE_BYTES], void **mapped)
{
    if (!ctx || !handle || !mapped) return fail(ctx, RTB_ERR_INVALID, "rtb_ipc_open: null argument");
    *mapped = nullptr;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    CUDA_TRY(ctx, cudaIpcOpenMemHandle(mapped, h, cudaIpcMemLazyEnablePeerAccess)); // maps the owner's memory; peer access over NVLink as needed
    return RTB_OK;
}

extern "C" int rtb_ipc_close(rtb_ctx *ctx, void *mapped)
{
    if (!ctx) return fail(ctx, RTB_ERR_INVALID, "rtb_ipc_close: null context");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (mapped)
    {
        if (ctx->frame_pending) CUDA_TRY(ctx, cudaEventSynchronize(ctx->last_frame)); // no frame may still store into it
        CUDA_TRY(ctx, cudaIpcCloseMemHandle(mapped));
    }
    return RTB_OK;
}

struct rtb_multi
{
    std::vector<rtb_ctx *> ctx;
    void *frame = nullptr; // page-locked frame for callers whose buffer is pageable
    size_t frame_bytes = 0;
    rtb_progress_fn progress = nullptr;
    void *progress_user = nullptr;
    std::string error;
    WorkerPool pool;
};
struct rtb_multi_scene { std::vector<rtb_scene *> s; };

static int failMulti(rtb_multi *m, int code, const std::string &msg)
{
    if (m) m->error = msg;
    return fail(nullptr, code, msg);
}

extern "C" const char *rtb_multi_last_error(const rtb_multi *m) { return m ? m->error.c_str() : rtb_last_error(nullptr); }
extern "C" int rtb_multi_count(const rtb_multi *m) { return m ? (int)m->ctx.size() : 0; }
extern "C" rtb_ctx *rtb_multi_ctx(rtb_multi *m, int i) { return (m && i >= 0 && i < (int)m->ctx.size()) ? m->ctx[(size_t)i] : nullptr; }

extern "C" int rtb_multi_shutdown(rtb_multi *m)
{
    if (!m) return RTB_OK;
    m->pool.shutdown();
    // the first context's staging ring is read by the other contexts' streams: they drain (rtb_shutdown) before it is freed
    for (size_t i = m->ctx.size(); i-- > 0;) rtb_shutdown(m->ctx[i]);
    if (m->frame) cudaFreeHost(m->frame);
    delete m;
    return RTB_OK;
}

extern "C" int rtb_multi_init(int n_devices, const int *devices, rtb_multi **out)
{
    if (!out) return fail(nullptr, RTB_ERR_INVALID, "rtb_multi_init: null output pointer");
    *out = nullptr;
    if (n_devices <= 0 || n_devices > 64) return fail(nullptr, RTB_ERR_INVALID, "rtb_multi_init: device count out of range");
    rtb_multi *m = new rtb_multi();
    for (int i = 0; i < n_devices; i++)
    {
        rtb_ctx *c = nullptr;
        const int rc = rtb_init(devices ? devices[i] : i, &c);
        if (rc != RTB_OK) { rtb_multi_shutdown(m); return rc; }
        m->ctx.push_back(c);
        if (i > 0) m->ctx[0]->stage_readers.push_back(c);
    }
    m->pool.start(n_devices - 1);
    *out = m;
    return RTB_OK;
}

extern "C" int rtb_multi_set_progress(rtb_multi *m, rtb_progress_fn fn, void *user)
{
    if (!m) return fail(nullptr, RTB_ERR_INVALID, "rtb_multi_set_progress: null argument");
    for (rtb_ctx *c : m->ctx)
    { // the contexts only provide the side stream and the read-back word; the reporting is done here, over all devices
        const int rc = rtb_set_progress(c, fn, user);
        if (rc != RTB_OK) return rc;
        c->progress = nullptr;
    }
    m->progress = fn;
    m->progress_user = user;
    return RTB_OK;
}

extern "C" int rtb_multi_scene_free(rtb_multi *m, rtb_multi_scene *s)
{
    if (!s) return RTB_OK;
    for (size_t i = 0; i < s->s.size(); i++)
        if (s->s[i]) rtb_scene_free(m && i < m->ctx.size() ? m->ctx[i] : nullptr, s->s[i]);
    delete s;
    return RTB_OK;
}

extern "C" int rtb_multi_scene_upload(rtb_multi *m, const rtb_flat_scene *flat, rtb_multi_scene **out)
{
    if (!m || !flat || !out) return failMulti(m, RTB_ERR_INVALID, "rtb_multi_scene_upload: null argument");
    *out = nullptr;
    const size_t n = m->ctx.size();
    rtb_multi_scene *s = new rtb_multi_scene();
    s->s.assign(n, nullptr);
    std::vector<int> rc(n, RTB_OK);
    // All devices upload side by side.  The calling thread runs the first device's upload, which validates the flat scene
    // (whole-stream index / structure checks on worker threads of its own) and stages every stream ONCE in its page-locked
    // ring; the other devices' uploads run on the pool's threads a step behind it: they take the staged bytes (StageShare)
    // for their own H2D copies and packing kernels, and wait for the verdict of the checks before anything indexes with the
    // checked streams.  8 B200: 1.63 ms (first device, then the replicas side by side with a staging pass each) -> 0.42-0.66 ms.
    StageShare share;
    if (n > 1)
    {
        // the whole upload in one stretch of the ring: a wrap in the middle would reuse bytes the replicas still copy from
        rtb_ctx *c0 = m->ctx[0];
        const size_t bound = stagedBytesBound(flat);
        if (c0->stage_used + bound > c0->stage_cap)
        {
            char *unused = nullptr;
            c0->stage_used = c0->stage_cap; // take stageReserve's drain-and-restart (or grow) path now
            cudaSetDevice(c0->device);
            const int e = stageReserve(c0, bound, &unused);
            if (e != RTB_OK) { delete s; return failMulti(m, e, c0->error); }
            c0->stage_used = 0;
        }
        for (size_t i = 0; i < n; i++)
        {
            m->ctx[i]->share = &share;
            m->ctx[i]->share_producer = i == 0;
            m->ctx[i]->share_next = 0;
        }
    }
    const std::function<void(int)> upload = [&](int i) {
        rc[(size_t)i] = sceneUpload(m->ctx[(size_t)i], flat, &s->s[(size_t)i], i == 0);
        if (i == 0 && rc[0] != RTB_OK) share.verdict.store(-1, std::memory_order_release); // releases the replicas
    };
    m->pool.run(upload);
    for (size_t i = 0; i < n; i++) m->ctx[i]->share = nullptr;
    for (size_t i = 0; i < n; i++)
        if (rc[i] != RTB_OK)
        {
            const size_t blame = rc[0] != RTB_OK ? 0 : i; // a replica released by a failed first upload only reports that
            const std::string msg = std::string("device ") + std::to_string(m->ctx[blame]->device) + ": " + m->ctx[blame]->error;
            const int code = rc[blame];
            rtb_multi_scene_free(m, s);
            return failMulti(m, code, msg);
        }
    *out = s;
    return RTB_OK;
}

extern "C" int rtb_multi_scene_mesh_update(rtb_multi *m, rtb_multi_scene *s, int32_t mesh_index, const float *tri, int64_t n,
                                           int32_t flags)
{
    if (!m || !s || !tri || s->s.size() != m->ctx.size()) return failMulti(m, RTB_ERR_INVALID, "rtb_multi_scene_mesh_update: null argument");
    rtb_ctx *c0 = m->ctx[0];
    std::vector<int> recs; // every device holds the same records: the checks on the first one hold for all
    int rc = meshUpdateRecords(c0, s->s[0], mesh_index, n, flags, recs);
    if (rc != RTB_OK) return failMulti(m, rc, c0->error);
    if (cudaSetDevice(c0->device) != cudaSuccess) return failMulti(m, RTB_ERR_CUDA, "rtb_multi_scene_mesh_update: cudaSetDevice failed");
    cudaPointerAttributes attr;
    const bool onDevice = cudaPointerGetAttributes(&attr, tri) == cudaSuccess &&
                          (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged);
    cudaGetLastError();
    if (onDevice) return failMulti(m, RTB_ERR_INVALID, "rtb_multi_scene_mesh_update: the records must be host memory (not device or managed)");
    // staged once, in the first context's ring: every device copies from it (the ring is reused only after they all drained)
    const size_t bytes = (size_t)n * 12 * sizeof(float);
    char *staged = nullptr;
    if ((rc = stageReserve(c0, bytes, &staged)) != RTB_OK) return failMulti(m, rc, c0->error);
    memcpy(staged, tri, bytes);
    for (size_t i = 0; i < m->ctx.size(); i++)
    {
        rtb_ctx *c = m->ctx[i];
        if (cudaSetDevice(c->device) != cudaSuccess) return failMulti(m, RTB_ERR_CUDA, "rtb_multi_scene_mesh_update: cudaSetDevice failed");
        if ((rc = meshUpdateEnqueue(c, s->s[i], recs, (const float *)staged, true, flags, c->stream)) != RTB_OK)
            return failMulti(m, rc, "device " + std::to_string(c->device) + ": " + c->error);
    }
    return RTB_OK;
}

extern "C" int64_t rtb_multi_scene_upload_bytes(const rtb_multi_scene *s)
{
    int64_t total = 0;
    if (s) for (const rtb_scene *x : s->s) total += rtb_scene_upload_bytes(x);
    return total;
}

extern "C" int rtb_multi_render(rtb_multi *m, const rtb_multi_scene *scene, const rtb_camera *cam, const rtb_render_setting *setting,
                                const rtb_frame *frame, void *rgb_out, rtb_stats *stats)
{
    if (!m || !scene || !cam || !setting || !frame || !rgb_out) return failMulti(m, RTB_ERR_INVALID, "rtb_multi_render: null argument");
    const int n = (int)m->ctx.size();
    if ((int)scene->s.size() != n) return failMulti(m, RTB_ERR_INVALID, "rtb_multi_render: the scene belongs to another device set");
    rtb_frame fr = *frame;
    fr.rank = 0; fr.world = n;
    if (fr.row_block <= 0) fr.row_block = 8;
    // up to 4 devices the heavy row blocks around the vanishing point already land on different devices; above, narrow
    // column blocks give every device the same mix of tiles (DESIGN.md section 6)
    if (n < 5 || fr.width % (n * 32) != 0) { if (fr.col_block > 0 && (fr.col_block % 8 != 0 || fr.width % ((int64_t)n * fr.col_block) != 0)) fr.col_block = 0; }
    else if (fr.col_block <= 0) fr.col_block = 32;
    if (n > 1) fr.layout |= RTB_LAYOUT_GLOBAL;
    std::vector<FrameParams> F((size_t)n);
    for (int i = 0; i < n; i++)
    {
        fr.rank = i;
        const int rc = makeFrame(m->ctx[(size_t)i], scene->s[(size_t)i], cam, setting, &fr, F[(size_t)i]);
        if (rc != RTB_OK) return failMulti(m, rc, m->ctx[(size_t)i]->error);
        if (n == 1) F[(size_t)i].global_out = 0;
    }
    if (F[0].cost_map) return failMulti(m, RTB_ERR_UNSUPPORTED, "rtb_multi_render: no cost maps");
    const size_t bytes = frameBytes(F[0]);
    cudaSetDevice(m->ctx[0]->device);
    float *alias = hostAlias(rgb_out);
    bool staged = false;
    if (!alias)
    { // pageable caller buffer: the devices store into a page-locked frame of the library, one host copy follows
        if (bytes > m->frame_bytes)
        {
            for (rtb_ctx *c : m->ctx) if (c->frame_pending) { cudaSetDevice(c->device); cudaEventSynchronize(c->last_frame); }
            if (m->frame) cudaFreeHost(m->frame);
            m->frame = nullptr; m->frame_bytes = 0;
            if (cudaHostAlloc(&m->frame, bytes, cudaHostAllocPortable) != cudaSuccess) return failMulti(m, RTB_ERR_OOM, "rtb_multi_render: cannot allocate the page-locked frame");
            m->frame_bytes = bytes;
        }
        alias = hostAlias(m->frame);
        if (!alias) return failMulti(m, RTB_ERR_CUDA, "rtb_multi_render: page-locked frame is not device-accessible");
        staged = true;
    }
    std::vector<PendingFrame> P((size_t)n);
    int rc = RTB_OK;
    { // every device's launch sequence (~15 runtime calls) on its own thread: the last device starts with the first
        std::vector<int> rcs((size_t)n, RTB_OK);
        const std::function<void(int)> launch = [&](int i) {
            rtb_frame fi = fr;
            fi.rank = i;
            rcs[(size_t)i] = renderLaunch(m->ctx[(size_t)i], scene->s[(size_t)i], F[(size_t)i], &fi, alias, m->ctx[(size_t)i]->stream, true, nullptr, true, P[(size_t)i]);
        };
        m->pool.run(launch);
        for (int i = 0; i < n; i++)
            if (rcs[(size_t)i] != RTB_OK && rc == RTB_OK) { rc = rcs[(size_t)i]; m->error = m->ctx[(size_t)i]->error; }
    }
    if (rc == RTB_OK && m->progress) pollProgress(m->ctx.data(), P.data(), n, m->progress, m->progress_user);
    rtb_stats total;
    memset(&total, 0, sizeof(total));
    for (int i = 0; i < n; i++)
    { // every queued frame is waited for, whatever happened to the others
        rtb_stats st;
        const int rf = renderFinish(m->ctx[(size_t)i], P[(size_t)i], &st, false);
        if (rf != RTB_OK && rc == RTB_OK) { rc = rf; m->error = m->ctx[(size_t)i]->error; }
        total.n_rays += st.n_rays; total.n_tri_tests += st.n_tri_tests; total.n_steps += st.n_steps; total.n_local_rows += st.n_local_rows;
        total.n_launches += st.n_launches;
        if (st.kernel_ms > total.kernel_ms) total.kernel_ms = st.kernel_ms;
        if (st.total_ms > total.total_ms) total.total_ms = st.total_ms;
    }
    if (rc != RTB_OK) return fail(nullptr, rc, m->error);
    if (staged) memcpy(rgb_out, m->frame, bytes);
    if (stats) *stats = total;
    return RTB_OK;
}

extern "C" int rtb_host_alloc(size_t bytes, void **out)
{
    if (!out) return fail(nullptr, RTB_ERR_INVALID, "rtb_host_alloc: null output pointer");
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable); // every device of the process may store into it
    if (e != cudaSuccess) return fail(nullptr, RTB_ERR_CUDA, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
    return RTB_OK;
}

extern "C" int rtb_host_register(void *p, size_t bytes)
{
    if (!p || !bytes) return fail(nullptr, RTB_ERR_INVALID, "rtb_host_register: null range");
    const cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(nullptr, RTB_ERR_CUDA, std::string("cudaHostRegister: ") + cudaGetErrorString(e)); }
    return RTB_OK;
}

extern "C" int rtb_host_unregister(void *p)
{
    if (!p) return RTB_OK;
    const cudaError_t e = cudaHostUnregister(p);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(nullptr, RTB_ERR_CUDA, std::string("cudaHostUnregister: ") + cudaGetErrorString(e)); }
    return RTB_OK;
}

extern "C" int rtb_host_free(void *p)
{
    if (p) cudaFreeHost(p);
    return RTB_OK;
}

extern "C" int rtb_unshard_device(rtb_ctx *ctx, const void *gathered, void *image, int32_t width, int32_t height,
                                  int32_t world, int32_t row_block, int64_t rows_per_rank, void *stream)
{
    if (!ctx || !gathered || !image || width <= 0 || height <= 0 || world <= 0 || row_block <= 0 || rows_per_rank <= 0)
        return fail(ctx, RTB_ERR_INVALID, "rtb_unshard_device: bad argument");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t rowFloats = (size_t)width * 3;
    unsigned int bx = (unsigned int)((rowFloats / 4 + 255) / 256);
    if (bx == 0) bx = 1;
    if (bx > 8) bx = 8;
    k_unshard<<<dim3(bx, height), 256, 0, stream ? (cudaStream_t)stream : ctx->stream>>>(
        (const float *)gathered, (float *)image, width, height, world, row_block, (int)rows_per_rank);
    CUDA_TRY(ctx, cudaGetLastError());
    return RTB_OK;
}

extern "C" int rtb_unshard_cols_device(rtb_ctx *ctx, const void *gathered, void *image, int32_t width, int32_t height,
                                       int32_t world, int32_t row_block, int32_t col_block, void *stream)
{
    if (!ctx || !gathered || !image || width <= 0 || height <= 0 || world <= 0 || row_block <= 0 || col_block <= 0 || col_block % 8 != 0 ||
        width % ((int64_t)world * col_block) != 0)
        return fail(ctx, RTB_ERR_INVALID, "rtb_unshard_cols_device: bad argument");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    unsigned int bx = (unsigned int)(((size_t)width * 3 / 4 + 255) / 256);
    if (bx == 0) bx = 1;
    if (bx > 8) bx = 8;
    k_unshard_cols<<<dim3(bx, height), 256, 0, stream ? (cudaStream_t)stream : ctx->stream>>>(
        (const float *)gathered, (float *)image, width, height, world, row_block, col_block);
    CUDA_TRY(ctx, cudaGetLastError());
    return RTB_OK;
}

extern "C" int rtb_scatter_shard_device(rtb_ctx *ctx, const void *local, void *frame_buffer, const rtb_frame *frame, void *stream)
{
    if (!ctx || !local || !frame_buffer || !frame) return fail(ctx, RTB_ERR_INVALID, "rtb_scatter_shard_device: null argument");
    rtb_frame plain = *frame;
    plain.layout = RTB_LAYOUT_ROWMAJOR;
    const int64_t rows = rtb_shard_rows(&plain), lw = rtb_shard_width(&plain);
    if (rows < 0 || (frame->layout & (RTB_LAYOUT_REFERENCE | RTB_OUTPUT_RGB8 | RTB_OUTPUT_MOMENTS)))
        return fail(ctx, RTB_ERR_INVALID, "rtb_scatter_shard_device: bad shard, or not a row-major float frame");
    const int world = frame->world > 0 ? frame->world : 1, cb = colSharded(frame) ? frame->col_block : 0;
    if (lw % 4 != 0 || (cb && (cb * 3) % 4 != 0) || frame->width % 4 != 0 || ((uintptr_t)local & 15u) || ((uintptr_t)frame_buffer & 15u))
        return fail(ctx, RTB_ERR_UNSUPPORTED, "rtb_scatter_shard_device: widths must be multiples of 4 pixels and the buffers 16-byte aligned");
    if (rows == 0) return RTB_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    unsigned int bx = (unsigned int)((lw * 3 / 4 + 255) / 256);
    if (bx == 0) bx = 1;
    if (bx > 8) bx = 8;
    k_scatter_shard<<<dim3(bx, (unsigned int)rows), 256, 0, stream ? (cudaStream_t)stream : ctx->stream>>>(
        (const float *)local, (float *)frame_buffer, frame->width, frame->height, world, frame->rank, normRowBlock(frame), cb, (int)lw, (int)rows);
    CUDA_TRY(ctx, cudaGetLastError());
    return RTB_OK;
}

// ---- parity hooks -----------------------------------------------------------------------------
template <class T> struct DevBuf
{
    T *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t n) { return cudaMalloc(&p, (n ? n : 1) * sizeof(T)); }
};

extern "C" int rtb_trace_primary(rtb_ctx *ctx, const rtb_scene *scene, const rtb_camera *cam, int32_t width, int32_t height,
                                 int32_t *hit_id, float *hit_t, int32_t *seq_len, uint64_t *seq_hash, int32_t *seq_buf,
                                 int32_t seq_cap)
{
    if (!ctx || !scene || !cam || width <= 0 || height <= 0) return fail(ctx, RTB_ERR_INVALID, "rtb_trace_primary: bad argument");
    if (seq_buf && seq_cap <= 0) return fail(ctx, RTB_ERR_INVALID, "rtb_trace_primary: seq_buf needs seq_cap > 0");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    FrameParams F;
    memset(&F, 0, sizeof(F));
    F.cam = *cam; F.width = width; F.height = height; F.rank = 0; F.world = 1; F.row_block = 8; F.n_local_rows = height; F.local_width = width;
    F.tiles_x = (width + RTB_TILE_W - 1) / RTB_TILE_W;
    F.n_tiles = F.tiles_x * ((height + RTB_TILE_H - 1) / RTB_TILE_H);
    F.warps_per_cta = RTB_CTA_THREADS / 32;
    const size_t n = (size_t)width * height;
    DevBuf<int> d_id, d_len, d_buf;
    DevBuf<float> d_t;
    DevBuf<unsigned long long> d_hash;
    if (hit_id) CUDA_TRY(ctx, d_id.alloc(n));
    if (hit_t) CUDA_TRY(ctx, d_t.alloc(n));
    if (seq_len) CUDA_TRY(ctx, d_len.alloc(n));
    if (seq_hash) CUDA_TRY(ctx, d_hash.alloc(n));
    if (seq_buf) CUDA_TRY(ctx, d_buf.alloc(n * seq_cap));
    const dim3 grid((unsigned int)((F.n_tiles + RTB_CTA_THREADS / 32 - 1) / (RTB_CTA_THREADS / 32)));
    if (scene->has_mesh) k_trace_primary<true><<<grid, RTB_CTA_THREADS, 0, ctx->stream>>>(scene->d, F, d_id.p, d_t.p, d_len.p, d_hash.p, d_buf.p, seq_cap);
    else k_trace_primary<<<grid, RTB_CTA_THREADS, 0, ctx->stream>>>(scene->d, F, d_id.p, d_t.p, d_len.p, d_hash.p, d_buf.p, seq_cap);
    CUDA_TRY(ctx, cudaGetLastError());
    if (hit_id) CUDA_TRY(ctx, cudaMemcpyAsync(hit_id, d_id.p, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (hit_t) CUDA_TRY(ctx, cudaMemcpyAsync(hit_t, d_t.p, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (seq_len) CUDA_TRY(ctx, cudaMemcpyAsync(seq_len, d_len.p, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (seq_hash) CUDA_TRY(ctx, cudaMemcpyAsync(seq_hash, d_hash.p, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (seq_buf) CUDA_TRY(ctx, cudaMemcpyAsync(seq_buf, d_buf.p, n * seq_cap * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return RTB_OK;
}

static void launchQuery(const rtb_scene *scene, const QueryParams &Q, bool any, cudaStream_t st)
{
    const unsigned int blocks = (unsigned int)((Q.n + RTB_CTA_THREADS - 1) / RTB_CTA_THREADS);
    if (scene->has_mesh)
    {
        if (any) k_query_rays<true, true><<<blocks, RTB_CTA_THREADS, 0, st>>>(scene->d, Q);
        else k_query_rays<true, false><<<blocks, RTB_CTA_THREADS, 0, st>>>(scene->d, Q);
    }
    else if (any) k_query_rays<false, true><<<blocks, RTB_CTA_THREADS, 0, st>>>(scene->d, Q);
    else k_query_rays<false, false><<<blocks, RTB_CTA_THREADS, 0, st>>>(scene->d, Q);
}

// A caller's buffer for rtb_query_rays / rtb_query_points / rtb_query_winding / rtb_query_triangles: memory of the context's device or managed memory, `align`-byte aligned
static bool deviceBuffer(const rtb_ctx *ctx, const void *p, uintptr_t align)
{
    cudaPointerAttributes attr;
    const bool known = cudaPointerGetAttributes(&attr, p) == cudaSuccess;
    cudaGetLastError();
    if (!known || ((uintptr_t)p & (align - 1))) return false;
    return attr.type == cudaMemoryTypeManaged || (attr.type == cudaMemoryTypeDevice && attr.device == ctx->device);
}

// The part rtb_query_rays, rtb_query_points, rtb_query_winding and rtb_query_triangles share.  Before the launch (queryBegin): the buffer checks -- the input array
// `in` (required) and the optional bound and outputs `bufs` -- and the ordering of the caller's stream behind the scene's
// upload / updates and behind the last query on another stream.  After it (queryEnd): query_use recorded on that stream.
// Every check comes before anything is enqueued.
static int queryBegin(rtb_ctx *ctx, const rtb_scene *scene, const char *fn, const char *in_name, const void *in, uintptr_t in_align,
                      const void *const bufs[6], const uintptr_t align[6], const char *bufs_name, void *stream, cudaStream_t &st)
{
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (!in || !deviceBuffer(ctx, in, in_align))
        return fail(ctx, RTB_ERR_INVALID, std::string(fn) + ": " + in_name + " must be " + std::to_string(in_align) +
                                              "-byte aligned memory of the context's device or managed memory");
    for (int b = 0; b < 6; b++)
        if (bufs[b] && !deviceBuffer(ctx, bufs[b], align[b]))
            return fail(ctx, RTB_ERR_INVALID, std::string(fn) + ": " + bufs_name +
                                                  " must be aligned memory of the context's device or managed memory");
    st = stream ? (cudaStream_t)stream : ctx->stream;
    if (st != ctx->stream) CUDA_TRY(ctx, cudaStreamWaitEvent(st, scene->ready, 0)); // uploads and updates run on ctx->stream
    if (scene->queried && st != scene->query_stream) CUDA_TRY(ctx, cudaStreamWaitEvent(st, scene->query_use, 0));
    return RTB_OK;
}

static int queryEnd(rtb_ctx *ctx, const rtb_scene *scene, cudaStream_t st)
{
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaEventRecord(scene->query_use, st));
    scene->query_stream = st;
    scene->queried = true;
    return RTB_OK;
}

extern "C" int rtb_query_rays(rtb_ctx *ctx, const rtb_scene *scene, int64_t n, const float *rays, const float *tmax, float tmax_all,
                              int32_t flags, int32_t *hit_id, float *hit_t, float *position, float *normal, uint8_t *occluded,
                              void *stream)
{
    if (!ctx || !scene || n < 0) return fail(ctx, RTB_ERR_INVALID, "rtb_query_rays: bad argument");
    if (flags != RTB_QUERY_CLOSEST && flags != RTB_QUERY_ANY) return fail(ctx, RTB_ERR_INVALID, "rtb_query_rays: unknown flags");
    const bool any = flags == RTB_QUERY_ANY;
    if (any ? (!occluded || hit_id || hit_t || position || normal) : occluded != nullptr)
        return fail(ctx, RTB_ERR_INVALID, "rtb_query_rays: the outputs do not match the flags (ANY: occluded only; CLOSEST: no occluded)");
    if (n == 0) return RTB_OK;
    const void *bufs[6] = {tmax, hit_id, hit_t, position, normal, occluded};
    const uintptr_t align[6] = {4, 4, 4, 4, 4, 1};
    cudaStream_t st;
    const int rc = queryBegin(ctx, scene, "rtb_query_rays", "rays", rays, 8, bufs, align, "tmax and the outputs", stream, st);
    if (rc != RTB_OK) return rc;
    QueryParams Q = {};
    Q.n = (long long)n; Q.rays = rays; Q.tmax = tmax; Q.tmax_all = tmax_all;
    Q.hit_id = hit_id; Q.hit_t = hit_t; Q.position = position; Q.normal = normal; Q.occluded = occluded;
    launchQuery(scene, Q, any, st);
    return queryEnd(ctx, scene, st);
}

extern "C" int rtb_query_points(rtb_ctx *ctx, const rtb_scene *scene, int64_t n, const float *points, const float *rmax,
                                float rmax_all, int32_t flags, int32_t *hit_id, float *distance, float *position, float *normal,
                                uint8_t *near, void *stream)
{
    if (!ctx || !scene || n < 0) return fail(ctx, RTB_ERR_INVALID, "rtb_query_points: bad argument");
    if (flags != RTB_QUERY_CLOSEST && flags != RTB_QUERY_ANY) return fail(ctx, RTB_ERR_INVALID, "rtb_query_points: unknown flags");
    const bool any = flags == RTB_QUERY_ANY;
    if (any ? (!near || hit_id || distance || position || normal) : near != nullptr)
        return fail(ctx, RTB_ERR_INVALID, "rtb_query_points: the outputs do not match the flags (ANY: near only; CLOSEST: no near)");
    if (n == 0) return RTB_OK;
    const void *bufs[6] = {rmax, hit_id, distance, position, normal, near};
    const uintptr_t align[6] = {4, 4, 4, 4, 4, 1};
    cudaStream_t st;
    const int rc = queryBegin(ctx, scene, "rtb_query_points", "points", points, 4, bufs, align, "rmax and the outputs", stream, st);
    if (rc != RTB_OK) return rc;
    PointParams Q = {};
    Q.n = (long long)n; Q.points = points; Q.rmax = rmax; Q.rmax_all = rmax_all;
    Q.hit_id = hit_id; Q.distance = distance; Q.position = position; Q.normal = normal; Q.near = near;
    const unsigned int blocks = (unsigned int)((Q.n + RTB_CTA_THREADS - 1) / RTB_CTA_THREADS);
    if (any) k_query_points<true><<<blocks, RTB_CTA_THREADS, 0, st>>>(scene->d, Q);
    else k_query_points<false><<<blocks, RTB_CTA_THREADS, 0, st>>>(scene->d, Q);
    return queryEnd(ctx, scene, st);
}

extern "C" int rtb_query_winding(rtb_ctx *ctx, const rtb_scene *scene, int64_t n, const float *points, float beta, float *winding,
                                 uint8_t *inside, void *stream)
{
    if (!ctx || !scene || n < 0) return fail(ctx, RTB_ERR_INVALID, "rtb_query_winding: bad argument");
    if (!(beta >= 1.0f)) return fail(ctx, RTB_ERR_INVALID, "rtb_query_winding: beta must be >= 1 (+inf: exact)");
    if (!winding && !inside) return fail(ctx, RTB_ERR_INVALID, "rtb_query_winding: no output (winding and inside are both null)");
    if (!scene->mesh_prims.empty() && !scene->mesh_moments)
        return fail(ctx, RTB_ERR_INVALID, "rtb_query_winding: the scene has MESH records but no moments: call rtb_scene_mesh_moments first");
    if (n == 0) return RTB_OK;
    const void *bufs[6] = {winding, inside, nullptr, nullptr, nullptr, nullptr};
    const uintptr_t align[6] = {4, 1, 1, 1, 1, 1};
    cudaStream_t st;
    const int rc = queryBegin(ctx, scene, "rtb_query_winding", "points", points, 4, bufs, align, "the outputs", stream, st);
    if (rc != RTB_OK) return rc;
    WindingParams Q = {};
    Q.n = (long long)n; Q.points = points; Q.moments = scene->mesh_moments; Q.beta = beta;
    Q.winding = winding; Q.inside = inside;
    k_query_winding<<<(unsigned int)((Q.n + RTB_CTA_THREADS - 1) / RTB_CTA_THREADS), RTB_CTA_THREADS, 0, st>>>(scene->d, Q);
    return queryEnd(ctx, scene, st);
}

extern "C" int rtb_query_triangles(rtb_ctx *ctx, const rtb_scene *scene, int64_t n, const float *tris, int32_t flags, uint8_t *hit,
                                   int32_t *pairs, int64_t capacity, int64_t *count, void *stream)
{
    if (!ctx || !scene || n < 0 || n > INT32_MAX) return fail(ctx, RTB_ERR_INVALID, "rtb_query_triangles: bad argument (n must be in [0, INT32_MAX])");
    if (flags != RTB_QUERY_ANY && flags != RTB_QUERY_PAIRS) return fail(ctx, RTB_ERR_INVALID, "rtb_query_triangles: unknown flags");
    const bool any = flags == RTB_QUERY_ANY;
    if (capacity < 0 || (capacity > 0 && !pairs)) return fail(ctx, RTB_ERR_INVALID, "rtb_query_triangles: capacity < 0, or capacity > 0 without pairs");
    if (any ? (!hit || pairs || count || capacity) : (hit || !count))
        return fail(ctx, RTB_ERR_INVALID, "rtb_query_triangles: the outputs do not match the flags (ANY: hit only; PAIRS: count and pairs, no hit)");
    if (n == 0 && any) return RTB_OK;
    const void *bufs[6] = {hit, pairs, n ? count : nullptr, nullptr, nullptr, nullptr};
    const uintptr_t align[6] = {1, 8, 8, 1, 1, 1};
    cudaStream_t st;
    // n == 0 in PAIRS mode reads no triangles but still defines *count: the count stands in for the input
    const int rc = n ? queryBegin(ctx, scene, "rtb_query_triangles", "tris", tris, 16, bufs, align, "the outputs", stream, st)
                     : queryBegin(ctx, scene, "rtb_query_triangles", "count", count, 8, bufs, align, "the outputs", stream, st);
    if (rc != RTB_OK) return rc;
    if (!any) CUDA_TRY(ctx, cudaMemsetAsync(count, 0, sizeof(int64_t), st));
    if (n > 0)
    {
        TriQueryParams Q = {};
        Q.n = (long long)n; Q.tris = tris; Q.hit = hit; Q.pairs = reinterpret_cast<int2 *>(pairs); Q.capacity = (long long)capacity;
        Q.count = reinterpret_cast<unsigned long long *>(count);
        const unsigned int blocks = (unsigned int)((Q.n + RTB_CTA_THREADS - 1) / RTB_CTA_THREADS);
        if (any) k_query_triangles<true><<<blocks, RTB_CTA_THREADS, 0, st>>>(scene->d, Q);
        else k_query_triangles<false><<<blocks, RTB_CTA_THREADS, 0, st>>>(scene->d, Q);
    }
    return queryEnd(ctx, scene, st);
}

extern "C" int rtb_intersect_rays(rtb_ctx *ctx, const rtb_scene *scene, int64_t n, const float *rays, int32_t *hit_id,
                                  float *hit_t, float *position, float *normal)
{
    if (!ctx || !scene || n < 0 || (n > 0 && !rays)) return fail(ctx, RTB_ERR_INVALID, "rtb_intersect_rays: bad argument");
    if (n == 0) return RTB_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    DevBuf<float> d_rays, d_t, d_pos, d_nrm;
    DevBuf<int> d_id;
    CUDA_TRY(ctx, d_rays.alloc((size_t)n * 6));
    CUDA_TRY(ctx, cudaMemcpyAsync(d_rays.p, rays, (size_t)n * 6 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    if (hit_id) CUDA_TRY(ctx, d_id.alloc((size_t)n));
    if (hit_t) CUDA_TRY(ctx, d_t.alloc((size_t)n));
    if (position) CUDA_TRY(ctx, d_pos.alloc((size_t)n * 3));
    if (normal) CUDA_TRY(ctx, d_nrm.alloc((size_t)n * 3));
    QueryParams Q = {};
    Q.n = (long long)n; Q.rays = d_rays.p; Q.tmax_all = INFINITY;
    Q.hit_id = d_id.p; Q.hit_t = d_t.p; Q.position = d_pos.p; Q.normal = d_nrm.p;
    launchQuery(scene, Q, false, ctx->stream);
    CUDA_TRY(ctx, cudaGetLastError());
    if (hit_id) CUDA_TRY(ctx, cudaMemcpyAsync(hit_id, d_id.p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (hit_t) CUDA_TRY(ctx, cudaMemcpyAsync(hit_t, d_t.p, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (position) CUDA_TRY(ctx, cudaMemcpyAsync(position, d_pos.p, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (normal) CUDA_TRY(ctx, cudaMemcpyAsync(normal, d_nrm.p, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return RTB_OK;
}

extern "C" int rtb_bounce_rays(rtb_ctx *ctx, const rtb_scene *scene, int64_t n, const float *rays, int32_t max_depth,
                               int32_t *reached, int32_t *depth, int32_t *last_id, float *last_pos, int64_t *total_rays,
                               float *kernel_ms)
{
    if (!ctx || !scene || n < 0 || (n > 0 && !rays) || max_depth < 0) return fail(ctx, RTB_ERR_INVALID, "rtb_bounce_rays: bad argument");
    if (total_rays) *total_rays = 0;
    if (kernel_ms) *kernel_ms = 0;
    if (n == 0) return RTB_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    DevBuf<float> d_rays, d_pos;
    DevBuf<int> d_ok, d_depth, d_id;
    CUDA_TRY(ctx, d_rays.alloc((size_t)n * 6));
    CUDA_TRY(ctx, cudaMemcpyAsync(d_rays.p, rays, (size_t)n * 6 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    if (reached) CUDA_TRY(ctx, d_ok.alloc((size_t)n));
    if (depth) CUDA_TRY(ctx, d_depth.alloc((size_t)n));
    if (last_id) CUDA_TRY(ctx, d_id.alloc((size_t)n));
    if (last_pos) CUDA_TRY(ctx, d_pos.alloc((size_t)n * 3));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->d_counters, 0, sizeof(Counters), ctx->stream));
    // small batches (the reference program traces 1000 rays): one warp per ray; see k_bounce_rays
    const int accel = scene->d.accel;
    const bool walkable = scene->has_tunnel && (accel == RTB_ACCEL_REGULAR_GRID || accel == RTB_ACCEL_FLAT_GRID || accel == RTB_ACCEL_KD_MEDIAN || accel == RTB_ACCEL_KD_SAH);
    static const long long wideMax = (long long)tunable("RTB_BOUNCE_WIDE_MAX", 148 * 64 * 2); // up to two warps per resident warp slot
    const bool wide = walkable && n <= wideMax && !scene->has_mesh; // the warp-per-ray walk has no mesh walk
    // one lane per ray: the lanes pull rays from a queue (Counters::steps doubles as its head), the grid fills the device once
    const long long resident = 148ll * 16 * RTB_CTA_THREADS;
    const long long threads = wide ? n * 32 : (n < resident ? n : resident);
    const unsigned int blocks = (unsigned int)((threads + RTB_CTA_THREADS - 1) / RTB_CTA_THREADS);
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], ctx->stream));
    if (wide) k_bounce_rays<true><<<blocks, RTB_CTA_THREADS, 0, ctx->stream>>>(scene->d, (long long)n, d_rays.p, max_depth, d_ok.p, d_depth.p, d_id.p,
                                                                             d_pos.p, &ctx->d_counters->rays, &ctx->d_counters->steps);
    else if (scene->has_mesh)
        k_bounce_rays<false, true><<<blocks, RTB_CTA_THREADS, 0, ctx->stream>>>(scene->d, (long long)n, d_rays.p, max_depth, d_ok.p, d_depth.p, d_id.p,
                                                                              d_pos.p, &ctx->d_counters->rays, &ctx->d_counters->steps);
    else k_bounce_rays<false><<<blocks, RTB_CTA_THREADS, 0, ctx->stream>>>(scene->d, (long long)n, d_rays.p, max_depth, d_ok.p, d_depth.p, d_id.p,
                                                                           d_pos.p, &ctx->d_counters->rays, &ctx->d_counters->steps);
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[2], ctx->stream));
    CUDA_TRY(ctx, cudaEventRecord(scene->last_use, ctx->stream));
    if (reached) CUDA_TRY(ctx, cudaMemcpyAsync(reached, d_ok.p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (depth) CUDA_TRY(ctx, cudaMemcpyAsync(depth, d_depth.p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (last_id) CUDA_TRY(ctx, cudaMemcpyAsync(last_id, d_id.p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (last_pos) CUDA_TRY(ctx, cudaMemcpyAsync(last_pos, d_pos.p, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    unsigned long long total = 0;
    CUDA_TRY(ctx, cudaMemcpyAsync(&total, &ctx->d_counters->rays, sizeof(total), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (total_rays) *total_rays = (int64_t)total;
    if (kernel_ms) CUDA_TRY(ctx, cudaEventElapsedTime(kernel_ms, ctx->ev[1], ctx->ev[2]));
    return RTB_OK;
}

// ---- self-test of the packed rejection test -------------------------------------------------------------------
__device__ __forceinline__ float selftestUniform(unsigned long long &state)
{ // splitmix64 -> [0, 1)
    state += 0x9e3779b97f4a7c15ull;
    unsigned long long z = state;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    z ^= z >> 31;
    return (float)(z >> 40) * (1.0f / 16777216.0f);
}

__device__ __forceinline__ rtb_pre::PreTri selftestTriangle(unsigned long long &st, float &scale)
{
    scale = powf(10.0f, -3.0f + 7.0f * selftestUniform(st));
    const float aspect = powf(10.0f, -3.0f * selftestUniform(st));
    const float offset = selftestUniform(st) < 0.5f ? 0.0f : powf(10.0f, 5.0f * selftestUniform(st)) - 1.0f;
    float t[12];
    for (int k = 0; k < 3; k++) t[k] = offset * (k == 2 ? -1.0f : 1.0f) + scale * (selftestUniform(st) - 0.5f);
    for (int k = 0; k < 3; k++) t[3 + k] = t[k] + scale * (selftestUniform(st) - 0.5f);
    for (int k = 0; k < 3; k++) t[6 + k] = t[k] + scale * aspect * (selftestUniform(st) - 0.5f);
    t[9] = 0; t[10] = 1; t[11] = 0;
    return rtb_pre::makePreTri(t);
}

__global__ void k_selftest_pretest(long long n, unsigned long long seed, unsigned long long *mismatches, unsigned long long *rejected)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned long long st = seed * 0x2545f4914f6cdd1dull + (unsigned long long)i * 0x9e3779b97f4a7c15ull;
    float s0, s1;
    const rtb_pre::PreTri A = selftestTriangle(st, s0), B = selftestTriangle(st, s1);
    // a ray through a point near the boundary of A (B sees an unrelated ray: mostly rejects, sometimes not)
    const float be = selftestUniform(st) * 1.2f - 0.1f, ga = (selftestUniform(st) < 0.5f) ? (selftestUniform(st) - 0.5f) * 2e-3f : selftestUniform(st) * 1.2f - 0.1f;
    const float tx = A.ax - A.e1x * be - A.e2x * ga, ty = A.ay - A.e1y * be - A.e2y * ga, tz = A.az - A.e1z * be - A.e2z * ga;
    float dx = selftestUniform(st) - 0.5f, dy = selftestUniform(st) - 0.5f, dz = selftestUniform(st) - 0.5f;
    const float inv = 1.0f / sqrtf(dx * dx + dy * dy + dz * dz + 1e-30f);
    dx *= inv; dy *= inv; dz *= inv;
    const float dist = s0 * powf(10.0f, -2.0f + 5.0f * selftestUniform(st));
    const float ox = tx - dx * dist, oy = ty - dy * dist, oz = tz - dz * dist;
    const float dmx = rtb_pre::dirMax(dx, dy, dz);
    const float lo = selftestUniform(st) < 0.5f ? -FLT_MAX : dist * (1.0f - 1e-3f * selftestUniform(st));
    const float hi = selftestUniform(st) < 0.5f ? FLT_MAX : dist * (1.0f + 1e-3f * selftestUniform(st));
    const float Lp = rtb_pre::lowBound(lo), Hp = rtb_pre::highBound(hi, FLT_MAX);
    rtb_pre::PreTri2 P;
    P.ax = make_float2(A.ax, B.ax); P.ay = make_float2(A.ay, B.ay); P.az = make_float2(A.az, B.az); P.a1e = make_float2(A.a1e, B.a1e);
    P.e1x = make_float2(A.e1x, B.e1x); P.e1y = make_float2(A.e1y, B.e1y); P.e1z = make_float2(A.e1z, B.e1z); P.ee = make_float2(A.ee, B.ee);
    P.e2x = make_float2(A.e2x, B.e2x); P.e2y = make_float2(A.e2y, B.e2y); P.e2z = make_float2(A.e2z, B.e2z);
    bool r0, r1, q0, q1;
    rtb_pre::sureReject2<true>(P, ox, oy, oz, dx, dy, dz, dmx, Lp, Hp, r0, r1);
    rtb_pre::sureReject2<false>(P, ox, oy, oz, dx, dy, dz, dmx, Lp, Hp, q0, q1);
    const bool s0h = rtb_pre::sureReject<true>(A, ox, oy, oz, dx, dy, dz, dmx, Lp, Hp), s1h = rtb_pre::sureReject<true>(B, ox, oy, oz, dx, dy, dz, dmx, Lp, Hp);
    const bool s0l = rtb_pre::sureReject<false>(A, ox, oy, oz, dx, dy, dz, dmx, Lp, Hp), s1l = rtb_pre::sureReject<false>(B, ox, oy, oz, dx, dy, dz, dmx, Lp, Hp);
    const unsigned int bad = (r0 != s0h) + (r1 != s1h) + (q0 != s0l) + (q1 != s1l);
    if (bad) atomicAdd(mismatches, (unsigned long long)bad);
    if (s0h) atomicAdd(rejected, 1ull);
}

extern "C" int rtb_selftest_pretest(rtb_ctx *ctx, int64_t n, uint64_t seed, int64_t *mismatches, int64_t *rejected)
{
    if (!ctx || n <= 0 || !mismatches || !rejected) return fail(ctx, RTB_ERR_INVALID, "rtb_selftest_pretest: bad argument");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    DevBuf<unsigned long long> d;
    CUDA_TRY(ctx, d.alloc(2));
    CUDA_TRY(ctx, cudaMemsetAsync(d.p, 0, 2 * sizeof(unsigned long long), ctx->stream));
    k_selftest_pretest<<<(unsigned int)((n + 255) / 256), 256, 0, ctx->stream>>>((long long)n, (unsigned long long)seed, d.p, d.p + 1);
    CUDA_TRY(ctx, cudaGetLastError());
    unsigned long long h[2] = {0, 0};
    CUDA_TRY(ctx, cudaMemcpyAsync(h, d.p, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *mismatches = (int64_t)h[0];
    *rejected = (int64_t)h[1];
    return RTB_OK;
}
