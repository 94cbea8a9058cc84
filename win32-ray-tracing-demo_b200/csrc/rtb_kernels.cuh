// rtb_kernels.cuh -- the render / trace kernels (sm_100a).
//
// Work decomposition: one thread owns one pixel, one WARP owns an 8x4 pixel tile (coherent primary
// rays, 4 x 96-byte row segments on the framebuffer store).  Tiles are the scheduling unit: warp w of
// the launch renders tile order[w].  Pixel cost on the tunnel scenes is extremely skewed -- the
// ~0.1 % of tiles around the vanishing point run 21-ray reflection chains that take ~60 x the median
// tile and, scheduled in raster order, ARE the kernel's critical path (profiles/r01_cost_map.md).
// So every render records the cycles each tile took and a counting sort turns that into a
// heaviest-first order for the next frame rendered with the same frame geometry (temporal
// coherence; the first frame of a geometry runs in raster order).  The order only changes
// scheduling: every pixel is computed by the same code whatever the order, so images are identical.
#pragma once
#include "rtb_device.cuh"

namespace rtb {

struct FrameParams
{
    rtb_camera cam;
    rtb_render_setting setting;
    int width, height, samples;
    int rank, world, row_block, layout;
    int col_block;   // > 0: column-block sharding (localToGlobal); 0: whole rows
    int local_width; // width of this rank's local image (= width unless col_block)
    int n_local_rows;
    int cost_map;
    int rgb8; // RTB_OUTPUT_RGB8
    int global_out; // RTB_LAYOUT_GLOBAL: `out` is the whole frame [height][width][3]; this rank stores its pixels at y * width + x
    int moments;    // RTB_OUTPUT_MOMENTS (Monte Carlo): six floats per pixel, sum and sum of squares of the per-sample radiance
    int sample_first, sample_end; // Monte Carlo: this launch renders samples [sample_first, sample_end) of `samples`
    int wide_store; // row-major output, 16-byte aligned rows: full tiles leave through storeTile()
    int group4;     // frames stored straight into page-locked HOST memory: the tile order is an order of GROUPS of four
                    // adjacent tiles, so a CTA of the throughput kernels holds one block of pixels and stores it in long
                    // segments (storeGroup); tier boundaries are multiples of four.
                    // 1: row-major frames, four horizontally adjacent tiles (order[4p + k] = 4g + k): a 32x4 block, four
                    //    384-byte row segments;  2: the reference's column-major frames (index = x * height + y), four
                    //    vertically adjacent tiles: an 8x16 block, eight 192-byte column segments
    int tiles_x, n_tiles;
    const unsigned int *order; // [n_tiles] tile ids, heaviest first; nullptr = raster order
    unsigned int *cost;        // [n_tiles] cycles >> 6 the throughput kernel last spent on each tile; may be nullptr
    const unsigned int *n_heavy; // number of leading entries of `order` that are latency-critical tiles (device value,
                                 // written by k_cost_offsets of the previous frame); use heavyCount()
    unsigned int n_wide;         // how many of those (the very heaviest) go to k_whitted_chain_wide (host value)
    unsigned int heavy_cap;      // upper bound of the latency-critical head the launch grids were sized for (host value)
    int skip_heavy;              // k_whitted_chain leaves those entries to k_whitted_chain_sm / _wide
    int record_cost;             // this launch records the cycles each of its tiles took (FrameParams::cost).  Only the
                                 // throughput kernel does: a tile rendered by a latency-optimised variant keeps the cost
                                 // it had when the throughput kernel last rendered it, so its rank -- and with it the
                                 // tier it is rendered by -- is stable from frame to frame (a cost recorded by a faster
                                 // variant would drop the tile out of its tier on the next frame, and back, forever)
    int split4;                  // this launch gives every tile to 4 warps of 8 lanes (one tile row each)
    int after_wide;              // this launch (k_whitted_chain_sm) starts at order[n_wide]
    int warps_per_cta;           // blockDim / 32
    // k_whitted_chain_oct (rtb_chain_oct.cuh): entries [item_base, min(item_end, heavyCount())) of the order
    unsigned int item_base, item_end;
    unsigned long long seed;
};

// Every kernel of a frame derives the tier boundaries from this one function, so each tile is rendered exactly
// once whatever the previous frame (possibly of another scene with the same frame geometry) left in *n_heavy
__device__ __forceinline__ unsigned int heavyCount(const FrameParams &F)
{
    unsigned int h = __ldg(F.n_heavy);
    if (F.group4) h = (h + 3u) & ~3u; // whole groups (a count left behind by a tile-granular frame may be anything)
    if (h > F.heavy_cap) h = F.heavy_cap;
    return h < F.n_wide ? F.n_wide : h;
}

#define RTB_CTA_THREADS 128 // 4 warp tiles per CTA: small CTAs retire (and free registers) early
#define RTB_TILE_W 8
#define RTB_TILE_H 4
#define RTB_COST_BUCKETS 128
#ifndef RTB_HEAVY_BUCKETS
#define RTB_HEAVY_BUCKETS 6 // quarter-octaves below the heaviest tile that still count as latency-critical (measured, scratch/perf2.py)
#endif
#ifndef RTB_HEAVY_FRACTION
#define RTB_HEAVY_FRACTION 128 // at most 1/128 of the tiles
#endif

// Local image -> frame.  A rank renders a LOCAL image of local_width x n_local_rows pixels (tiles, tile order and
// framebuffer slots are local); two ways of cutting the frame (rtb_frame.col_block):
//   rows    (col_block == 0): blocks of row_block rows dealt round-robin -- local row lr is global row
//           (lb * world + rank) * row_block + lr % row_block, lb = lr / row_block; x is unchanged;
//   columns (col_block > 0): every rank renders every row, and of block row by = y / row_block the column blocks bx
//           with (bx + by) % world == rank -- local column block c is global block c * world + (rank - by) mod world.
//           The tunnel frames concentrate their cost around the vanishing point; with rows, whichever ranks own those
//           few row blocks finish last, with narrow column blocks every rank holds the same mix of tiles.
// false when the local pixel lies outside the frame.
__device__ __forceinline__ bool localToGlobal(const FrameParams &F, int xl, int lr, int &x, int &y)
{
    if (F.col_block)
    {
        y = lr;
        const int by = lr / F.row_block;
        const int c = xl / F.col_block;
        int shift = (F.rank - by) % F.world;
        if (shift < 0) shift += F.world;
        x = (c * F.world + shift) * F.col_block + (xl - c * F.col_block);
        return xl < F.local_width && y < F.height; // x < width: width is a multiple of world * col_block
    }
    x = xl;
    const int lb = lr / F.row_block;
    y = (lb * F.world + F.rank) * F.row_block + (lr - lb * F.row_block);
    return x < F.width && lr < F.n_local_rows && y < F.height;
}

// warp -> tile -> (x, local row, global y); false when the thread has no pixel
__device__ __forceinline__ bool pixelOfThread(const FrameParams &F, int &x, int &lr, int &y, unsigned int &tile)
{
    const unsigned int w = blockIdx.x * (unsigned int)F.warps_per_cta + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    unsigned int item = F.split4 ? (w >> 2) : w; // index into the tile order
    if (F.after_wide) item += F.n_wide; // k_whitted_chain_sm: its tiles follow the wide kernel's
    tile = 0xffffffffu; // no tile: finishWarp records no cost
    if (item >= (unsigned int)F.n_tiles) return false;
    tile = F.order ? __ldg(F.order + item) : item;
    const int ty = tile / F.tiles_x, tx = tile - ty * F.tiles_x;
    if (F.split4 && lane >= 8) return false; // 8 active lanes: row (w & 3) of the tile
    const int xl = tx * RTB_TILE_W + (lane & 7);
    lr = ty * RTB_TILE_H + (F.split4 ? (int)(w & 3u) : (lane >> 3));
    return localToGlobal(F, xl, lr, x, y);
}

// framebuffer slot of global pixel (x, y) = local row lr
__device__ __forceinline__ size_t pixelSlot(const FrameParams &F, int x, int lr, int y)
{
    if (F.layout == RTB_LAYOUT_REFERENCE) return (size_t)x * F.height + y;
    if (F.global_out) return (size_t)y * F.width + x;
    int xl = x;
    if (F.col_block)
    {
        const int bx = x / F.col_block;
        xl = (bx / F.world) * F.col_block + (x - bx * F.col_block);
    }
    return (size_t)lr * F.local_width + xl;
}

// framebuffer store: float RGB, or the reference's 8-bit output stage (MainWindow.cpp:305-311)
__device__ __forceinline__ void storeColor(const FrameParams &F, float *out, int x, int lr, int y, V3 c)
{
    const size_t slot = pixelSlot(F, x, lr, y);
    if (F.rgb8)
    {
        unsigned char *o = reinterpret_cast<unsigned char *>(out) + 3 * slot;
        const float r = (c.x > 1.0f) ? 1.0f : c.x, g = (c.y > 1.0f) ? 1.0f : c.y, b = (c.z > 1.0f) ? 1.0f : c.z;
        o[0] = (unsigned char)f2i(r * 255); o[1] = (unsigned char)f2i(g * 255); o[2] = (unsigned char)f2i(b * 255);
    }
    else
    {
        float *o = out + 3 * slot;
        o[0] = c.x; o[1] = c.y; o[2] = c.z;
    }
}

// Whole-tile store of the throughput kernels.  A warp owns an 8x4 tile; written pixel by pixel each of its four
// 96-byte row segments leaves as 3 x 8 scalar stores that touch every 32-byte sector three times -- harmless in
// HBM, but when the kernels store straight into the caller's page-locked host frame every partial sector is its
// own PCIe write.  Here the 96 colour floats pass through 384 bytes of shared memory and leave as 24 128-bit
// stores, each sector written once (8-bit frames: 24 32-bit stores).  Returns false when the tile is ragged or
// the layout is not row-major / aligned: the caller then stores per pixel.
__device__ __forceinline__ bool storeTile(const FrameParams &F, float *out, unsigned int tile, bool active, V3 c, uint32_t *stage)
{
    if (!F.wide_store || !__all_sync(0xffffffffu, active)) return false;
    const int lane = threadIdx.x & 31;
    const int ty = tile / F.tiles_x, tx = tile - ty * F.tiles_x;
    const int row = lane / 6, j = lane - row * 6; // lanes 0..23: row 0..3, 16-byte (4-byte) chunk 0..5 of the row segment
    size_t rowSlot = (size_t)(ty * RTB_TILE_H + row) * F.local_width + (size_t)tx * RTB_TILE_W;
    if (F.global_out)
    { // the tile's row segment at its place in the whole frame: 8 consecutive pixels there too (blocks are multiples of 8)
        int xg, yg;
        localToGlobal(F, tx * RTB_TILE_W, ty * RTB_TILE_H + (row < RTB_TILE_H ? row : 0), xg, yg);
        rowSlot = (size_t)yg * F.width + xg;
    }
    if (F.rgb8)
    {
        unsigned char *sb = reinterpret_cast<unsigned char *>(stage);
        const float r = (c.x > 1.0f) ? 1.0f : c.x, g = (c.y > 1.0f) ? 1.0f : c.y, b = (c.z > 1.0f) ? 1.0f : c.z;
        sb[3 * lane + 0] = (unsigned char)f2i(r * 255); sb[3 * lane + 1] = (unsigned char)f2i(g * 255); sb[3 * lane + 2] = (unsigned char)f2i(b * 255);
        __syncwarp();
        if (lane < 24) *reinterpret_cast<uint32_t *>(reinterpret_cast<unsigned char *>(out) + 3 * rowSlot + 4 * j) = stage[lane];
    }
    else
    {
        float *sf = reinterpret_cast<float *>(stage);
        sf[3 * lane + 0] = c.x; sf[3 * lane + 1] = c.y; sf[3 * lane + 2] = c.z;
        __syncwarp();
        if (lane < 24) *reinterpret_cast<float4 *>(out + 3 * rowSlot + 4 * j) = reinterpret_cast<const float4 *>(stage)[lane];
    }
    return true;
}
#define RTB_TILE_STAGE_WORDS 96

// CTA-wide store of the throughput kernels for frames in page-locked HOST memory (FrameParams::group4).  Written tile by
// tile, every 96-byte row segment is its own PCIe write unless a neighbouring tile finishes at the same moment.  Measured on
// a B200 (tools/probes/pcie_store_probe.cu, a 3840x2880 float frame stored into host memory by an otherwise idle kernel):
// 96-byte segments reach 49.6 GB/s in raster order but 25.5 GB/s in any other order; 384-byte segments 52 GB/s in ANY order
// (the copy engine: 57 GB/s).  So the four warps of a CTA take four horizontally adjacent tiles (the order is an order of
// such groups), pass the 32x4 pixels through the CTA's staging memory and 96 threads store them as four 384-byte row
// segments of 128-bit stores (8-bit frames: four 96-byte segments of 32-bit stores).  4K SAH frame into host memory:
// 5.11 -> 4.85 ms (into HBM: 4.70), profiles/r02_group_store.log.
// The reference's own framebuffer order, colors[x * height + y] (MainWindow.cpp:276: what CudaRenderer::Render, the RenderProc
// drop-in, asks for), is column-major: a tile is eight 48-byte column pieces there, and written pixel by pixel into host memory
// the 4K SAH kernel took 9.9 ms.  For that layout a group is four VERTICALLY adjacent tiles, an 8x16-pixel block that leaves as
// eight 192-byte column segments.
// All threads of the CTA must call it.  false: group mode is off, a tile is ragged, or the CTA's tiles are not one group
// (an order inherited from a tile-granular frame) -- nothing was stored, the caller stores per tile.
__device__ __forceinline__ bool storeGroup(const FrameParams &F, float *out, unsigned int tile, bool active, V3 c,
                                           uint32_t (*stage)[RTB_TILE_STAGE_WORDS])
{
    if (!F.group4) return false; // uniform over the launch
    __shared__ unsigned int groupTile[RTB_CTA_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool vertical = F.group4 == 2;
    if (lane == 0) groupTile[warp] = tile;
    if (!__syncthreads_and(active && tile != 0xffffffffu)) return false;
    const unsigned int t0 = groupTile[0], step = vertical ? (unsigned int)F.tiles_x : 1u;
    const int ty = t0 / F.tiles_x, tx = t0 - ty * F.tiles_x;
    if (((vertical ? (unsigned int)ty : t0) & 3u) != 0u || groupTile[1] != t0 + step || groupTile[2] != t0 + 2u * step || groupTile[3] != t0 + 3u * step)
        return false; // uniform
    // the block's pixels in the order they leave: row-major blocks [4 rows][32 px][3], column-major blocks [8 columns][16 px][3]
    const int col = lane & 7, row = lane >> 3;
    const int at = vertical ? (col * 16 + warp * 4 + row) * 3 : 0; // (horizontal: per-tile staging, gathered by the storing threads)
    if (F.rgb8)
    {
        unsigned char *sb = vertical ? reinterpret_cast<unsigned char *>(stage[0]) + at : reinterpret_cast<unsigned char *>(stage[warp]) + 3 * lane;
        const float r = (c.x > 1.0f) ? 1.0f : c.x, g = (c.y > 1.0f) ? 1.0f : c.y, b = (c.z > 1.0f) ? 1.0f : c.z;
        sb[0] = (unsigned char)f2i(r * 255); sb[1] = (unsigned char)f2i(g * 255); sb[2] = (unsigned char)f2i(b * 255);
    }
    else
    {
        float *sf = vertical ? reinterpret_cast<float *>(stage[0]) + at : reinterpret_cast<float *>(stage[warp]) + 3 * lane;
        sf[0] = c.x; sf[1] = c.y; sf[2] = c.z;
    }
    __syncthreads();
    if (threadIdx.x < 96)
    {
        if (vertical)
        { // column k of the block, 16-byte (4-byte) chunk `seg` of its 192-byte (48-byte) segment
            const int k = threadIdx.x / 12, seg = threadIdx.x - k * 12;
            const size_t slot = (size_t)(tx * RTB_TILE_W + k) * F.height + (size_t)ty * RTB_TILE_H; // world == 1: local rows are frame rows
            if (F.rgb8)
                *reinterpret_cast<uint32_t *>(reinterpret_cast<unsigned char *>(out) + 3 * slot + 4 * seg) = stage[0][k * 12 + seg];
            else
                *reinterpret_cast<float4 *>(out + 3 * slot + 4 * seg) = reinterpret_cast<const float4 *>(stage[0])[k * 12 + seg];
        }
        else
        {
            const int r = threadIdx.x / 24, seg = threadIdx.x - r * 24; // 16-byte (4-byte) chunk `seg` of the group's row segment
            const int k = seg / 6, j = seg - k * 6;                     // tile k of the group, chunk j of that tile's row
            size_t rowSlot = (size_t)(ty * RTB_TILE_H + r) * F.local_width + (size_t)tx * RTB_TILE_W;
            if (F.global_out)
            { // a group is 32 consecutive pixels of the whole frame too (column blocks are multiples of 32 in group mode)
                int xg, yg;
                localToGlobal(F, tx * RTB_TILE_W, ty * RTB_TILE_H + r, xg, yg);
                rowSlot = (size_t)yg * F.width + xg;
            }
            if (F.rgb8)
                *reinterpret_cast<uint32_t *>(reinterpret_cast<unsigned char *>(out) + 3 * rowSlot + 4 * seg) = stage[k][r * 6 + j];
            else
                *reinterpret_cast<float4 *>(out + 3 * rowSlot + 4 * seg) = reinterpret_cast<const float4 *>(stage[k])[r * 6 + j];
        }
    }
    return true;
}

// per-warp epilogue: record the tile's cost, add the warp's counters to the frame totals
__device__ __forceinline__ void finishWarp(const FrameParams &F, Counters *g, unsigned int tile, long long t_start,
                                           unsigned int rays, unsigned int tris, unsigned int steps)
{
    __syncwarp();
    rays = __reduce_add_sync(0xffffffffu, rays);
    tris = __reduce_add_sync(0xffffffffu, tris);
    steps = __reduce_add_sync(0xffffffffu, steps);
    if ((threadIdx.x & 31) == 0)
    {
        if (F.record_cost && F.cost && tile != 0xffffffffu)
        {
            const long long dt = (clock64() - t_start) >> 6;
            F.cost[tile] = dt > 0xffffffffll ? 0xffffffffu : (unsigned int)dt; // one warp per tile in the recording launches
        }
        if (rays) atomicAdd(&g->rays, (unsigned long long)rays);
        if (tris) atomicAdd(&g->tris, (unsigned long long)tris);
        if (steps) atomicAdd(&g->steps, (unsigned long long)steps);
        // finished tiles (rtb_set_progress); a split4 launch gives a tile to four warps: the first one reports it
        if (tile != 0xffffffffu && (!F.split4 || ((blockIdx.x * (unsigned int)F.warps_per_cta + (threadIdx.x >> 5)) & 3u) == 0u)) atomicAdd(&g->tiles, 1ull);
    }
}

template <class Probe> struct ProbeCounts
{
    static __device__ __forceinline__ unsigned int tris(const Probe &) { return 0; }
    static __device__ __forceinline__ unsigned int steps(const Probe &) { return 0; }
};
template <> struct ProbeCounts<CountProbe>
{
    static __device__ __forceinline__ unsigned int tris(const CountProbe &p) { return p.tris; }
    static __device__ __forceinline__ unsigned int steps(const CountProbe &p) { return p.steps; }
};

// ---------------------------------------------------------------------------------------------
// Whitted, scenes without refractive materials: the recursion of reference MainWindow.cpp:69-143
// degenerates to a chain of reflections.  The chain is walked forward keeping (diffusive*d, r)
// per vertex, then folded back innermost-first so the float result is bit-identical to the
// recursive evaluation `diffusive*d + reflective*r + refractive*t`.
// ---------------------------------------------------------------------------------------------
#define RTB_MAX_DEPTH 100 // the reference's hard recursion cap (MainWindow.cpp:86)
// Fold stack of the chain kernels, in 16-byte entries of LOCAL memory per thread: one entry per reflective vertex, at
// most min(max_depth, RTB_MAX_DEPTH).  RenderSetting::Simple() (maxDepth 20: every tunnel preset) takes the short
// variant -- 384 bytes instead of 1,616 per thread, 151 k resident threads; deeper settings the long one.
#define RTB_FOLD_SHORT 24
#define RTB_FOLD_LONG (RTB_MAX_DEPTH + 1)
__host__ __device__ inline bool foldShortEnough(int max_depth) { return max_depth < RTB_FOLD_SHORT; }
#ifndef RTB_CHAIN_MIN_CTAS
#define RTB_CHAIN_MIN_CTAS 8 // 64 registers: measured best (5.9 ms vs 7.5 ms at 4) on the 4K SAH frame
#endif

// one pixel: walk the chain ray by ray (each ray a complete GeometrySet::intersect, `isect`), then fold
template <int FOLD, class Probe, class Isect>
__device__ __forceinline__ V3 chainWith(const DScene &S, const FrameParams &F, int x, int y, unsigned int &rays, Probe &pr, Isect isect)
{
    const float dx = 1.0f / F.height, dy = 1.0f / F.height; // MainWindow.cpp:254-255
    const float sx = (x + 0.5f) * dx, sy = 1 - (y + 0.5f) * dy;
    Ray r = generateRay(F.cam, sx, sy);
    float4 fold[FOLD];
    int n = 0, depth = 0;
    V3 c = v3(0, 0, 0); // value returned by the innermost call
    const V3 zero = v3(0, 0, 0);
    while (true)
    {
        rays++;
        Hit h;
        if (!isect(r, h)) break; // Color::Black()
        const rtb_material &m = S.mats[h.mat];
        const V3 nl = (dot(h.n, r.d) < 0) ? h.n : h.n * -1;
        const V3 local = matLocal(m, r, h.pos, h.n);
        if (++depth > F.setting.max_depth) break;
        if (depth > RTB_MAX_DEPTH) break;
        const V3 diffusive = (m.diffusiveness > 0) ? local : zero;
        const V3 term = diffusive * m.diffusiveness;
        if (m.reflectiveness > 0)
        {
            fold[n++] = make_float4(term.x, term.y, term.z, m.reflectiveness);
            const V3 v = r.d - nl * 2 * dot(nl, r.d);
            r.o = h.pos;
            r.d = v;
            continue;
        }
        c = term + zero * m.reflectiveness + zero * m.refractiveness;
        break;
    }
    while (n > 0)
    {
        const float4 f = fold[--n];
        c = v3(f.x, f.y, f.z) + c * f.w + zero * 0.0f;
    }
    return c;
}

template <int FOLD, bool MESH, class Probe>
__device__ __forceinline__ V3 chainPerRay(const DScene &S, const FrameParams &F, int x, int y, unsigned int &rays, Probe &pr)
{
    RayCtx ctx; // carried along the chain: trace() copies it to the reflected ray (MainWindow.cpp:105)
    ctx.inTunnel = 0; ctx.segment = -1;
    return chainWith<FOLD>(S, F, x, y, rays, pr, [&](const Ray &r, Hit &h) { return sceneIntersect<MESH>(S, r, h, pr, ctx); });
}

template <class Probe>
__device__ __forceinline__ void storePixel(const FrameParams &F, float *out, int x, int lr, int y, V3 c, long long t_start,
                                           unsigned int rays, const Probe &pr)
{
    if (F.cost_map && !F.rgb8)
    { // profiling aid: (thread cycles, rays, traversal steps + triangle tests) instead of the colour
        float *o = out + 3 * pixelSlot(F, x, lr, y);
        o[0] = (float)(clock64() - t_start); o[1] = (float)rays;
        o[2] = (float)(ProbeCounts<Probe>::tris(pr) + ProbeCounts<Probe>::steps(pr));
    }
    else storeColor(F, out, x, lr, y, c);
}

// MESH: scenes with RTB_PRIM_MESH records (rtb_device.cuh: sceneIntersectWith)
template <class Probe, int FOLD, bool MESH = false>
__global__ void __launch_bounds__(RTB_CTA_THREADS, RTB_CHAIN_MIN_CTAS)
k_whitted_chain(const __grid_constant__ DScene S, const __grid_constant__ FrameParams F, float *__restrict__ out,
                Counters *__restrict__ counters)
{
    int x, lr, y;
    unsigned int tile;
    const long long t_start = clock64();
    const bool active = pixelOfThread(F, x, lr, y, tile);
    unsigned int rays = 0;
    Probe pr;
    if (F.skip_heavy && blockIdx.x * (unsigned int)F.warps_per_cta + (threadIdx.x >> 5) < heavyCount(F)) return;
    __shared__ __align__(16) uint32_t stage[RTB_CTA_THREADS / 32][RTB_TILE_STAGE_WORDS];
    V3 c = v3(0, 0, 0);
    if (active) c = chainPerRay<FOLD, MESH>(S, F, x, y, rays, pr);
    if (!storeGroup(F, out, tile, active, c, stage) && !storeTile(F, out, tile, active, c, stage[threadIdx.x >> 5]) && active)
        storePixel(F, out, x, lr, y, c, t_start, rays, pr);
    finishWarp(F, counters, tile, t_start, rays, ProbeCounts<Probe>::tris(pr), ProbeCounts<Probe>::steps(pr));
}

// ---------------------------------------------------------------------------------------------
// Whitted, general scenes (refractive materials present): the ray tree of MainWindow.cpp:69-143
// is walked depth-first with an explicit stack of {ray, scalar weight, depth}.  All branch weights
// (reflectiveness, refractiveness*Re, refractiveness*Tr) are scalars, so a node contributes
// weight * diffusive * d.  Accumulation order differs from the recursion: results agree within
// ~1e-6 relative (the stated tolerance is 1e-5), not bit for bit.
// ---------------------------------------------------------------------------------------------
#define RTB_TREE_STACK 64 // live items <= 2*max_depth + 1
struct TreeItem { V3 o, d; float w; int depth; };

template <class Probe, bool MESH = false>
__global__ void __launch_bounds__(RTB_CTA_THREADS)
k_whitted_tree(const __grid_constant__ DScene S, const __grid_constant__ FrameParams F, float *__restrict__ out,
               Counters *__restrict__ counters)
{
    int x, lr, y;
    unsigned int tile;
    const long long t_start = clock64();
    const bool active = pixelOfThread(F, x, lr, y, tile);
    unsigned int rays = 0;
    Probe pr;
    if (active)
    {
        const float dx = 1.0f / F.height, dy = 1.0f / F.height;
        const float sx = (x + 0.5f) * dx, sy = 1 - (y + 0.5f) * dy;
        const Ray primary = generateRay(F.cam, sx, sy);
        const int cap = RTB_TREE_STACK;
        TreeItem stack[RTB_TREE_STACK];
        int sp = 0;
        stack[sp].o = primary.o; stack[sp].d = primary.d; stack[sp].w = 1.0f; stack[sp].depth = 0; sp++;
        V3 c = v3(0, 0, 0);
        while (sp > 0)
        {
            const TreeItem it = stack[--sp];
            Ray r; r.o = it.o; r.d = it.d;
            int depth = it.depth;
            rays++;
            Hit h;
            if (!sceneIntersect<MESH>(S, r, h, pr)) continue;
            const rtb_material &m = S.mats[h.mat];
            const V3 nl = (dot(h.n, r.d) < 0) ? h.n : h.n * -1;
            const V3 local = matLocal(m, r, h.pos, h.n);
            if (++depth > F.setting.max_depth) continue;
            if (depth > RTB_MAX_DEPTH) continue;
            if (m.diffusiveness > 0) c = c + local * (it.w * m.diffusiveness);
            if (sp + 3 > cap) continue; // excluded by rtb_render: max_depth <= (RTB_TREE_STACK - 3) / 2
            // children are pushed in reverse so they pop in the reference's order
            if (m.refractiveness > 0)
            {
                const Fresnel f = refraction(r, h.n, nl, m.refractive_index);
                const float wt = it.w * m.refractiveness;
                if (f.tir) { stack[sp].o = h.pos; stack[sp].d = f.refl; stack[sp].w = wt; stack[sp].depth = depth; sp++; }
                else
                {
                    stack[sp].o = h.pos; stack[sp].d = f.tdir; stack[sp].w = wt * f.Tr; stack[sp].depth = depth; sp++;
                    stack[sp].o = h.pos; stack[sp].d = f.refl; stack[sp].w = wt * f.Re; stack[sp].depth = depth; sp++;
                }
            }
            if (m.reflectiveness > 0)
            {
                stack[sp].o = h.pos; stack[sp].d = r.d - nl * 2 * dot(nl, r.d);
                stack[sp].w = it.w * m.reflectiveness; stack[sp].depth = depth; sp++;
            }
        }
        storeColor(F, out, x, lr, y, c);
    }
    finishWarp(F, counters, tile, t_start, rays, ProbeCounts<Probe>::tris(pr), ProbeCounts<Probe>::steps(pr));
}

// ---------------------------------------------------------------------------------------------
// Monte-Carlo path tracing -- reference MainWindow.cpp:145-249 (radiance) + 277-291 (sampling).
// The recursion is unrolled into throughput form: `emission + local.mult(child)` becomes
// L += T*emission; T *= local.  The two-ray refraction split (depth <= singleTracingDepth) pushes
// the reflected ray and continues with the transmitted one -- the order in which the g++ build of
// the reference consumes its random stream -- so with the counter-based stream the draws line up
// with oracle/rt_oracle.cpp's ORACLE_RNG_COUNTER mode one to one.
// ---------------------------------------------------------------------------------------------
#define RTB_MC_STACK 32
struct McItem { V3 o, d, T; int depth; };

#ifndef RTB_MC_MIN_CTAS
#define RTB_MC_MIN_CTAS 5 // 96 registers
#endif
#ifndef RTB_MC_REFERENCE_TRIG
#define RTB_MC_REFERENCE_TRIG 0 // 1: phi = acosf(r2), cosf(phi), sinf(phi), cosf(theta), sinf(theta) literally (MainWindow.cpp:190-197)
#endif

template <class Probe, bool MESH = false>
__global__ void __launch_bounds__(RTB_CTA_THREADS, RTB_MC_MIN_CTAS)
k_montecarlo(const __grid_constant__ DScene S, const __grid_constant__ FrameParams F, float *__restrict__ out,
             Counters *__restrict__ counters)
{
    // Materials are indexed by the HIT, i.e. per lane: out of the constant bank every distinct index is a pass of its own
    // (ncu: the address-divergence unit 33 % busy); shared memory serves them in one.
    __shared__ rtb_material smat[RTB_MAX_INLINE_MATS];
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(S.mats);
        uint32_t *dst = reinterpret_cast<uint32_t *>(smat);
        for (int i = threadIdx.x; i < S.n_materials * (int)(sizeof(rtb_material) / 4); i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    int x, lr, y;
    unsigned int tile;
    const long long t_start = clock64();
    const bool active = pixelOfThread(F, x, lr, y, tile);
    unsigned int rays = 0;
    Probe pr;
    if (active)
    {
        const float dx = 1.0f / F.height, dy = 1.0f / F.height;
        const float PI_F = 3.14159265359f; // Vector.h:8
        const float inv = 1.0f / F.samples;
        V3 acc = v3(0, 0, 0);
        V3 sum = v3(0, 0, 0), sumsq = v3(0, 0, 0); // RTB_OUTPUT_MOMENTS: plain sums over this launch's samples
        McItem stack[RTB_MC_STACK];
        // ONE loop over ray segments: a lane whose path has ended accumulates the sample and starts its next
        // sample in the same iteration, so the warp never waits at a per-sample reconvergence point for its
        // longest path (Russian roulette makes path lengths 2..30; with a per-sample loop SIMT efficiency
        // was ~30 %).  Per-sample arithmetic and the accumulation order are unchanged.
        int s = F.sample_first, depth = 0, sp = 0; // a sample shard renders [sample_first, sample_end) of F.samples
        bool fresh = true;
        const uint32_t pixel = (uint32_t)(y * F.width + x);
        uint32_t block = 0; // Philox block of the next ray of this sample
        Ray r;
        r.o = v3(0, 0, 0); r.d = v3(0, 0, 1);
        V3 L = v3(0, 0, 0), T = v3(1, 1, 1);
        while (s < F.sample_end)
        {
            if (fresh)
            {
                const uint4 j = philoxBlock(pixel, (uint32_t)s, 0u, F.seed);
                const float sx = (x + uniform01(j.x)) * dx, sy = 1 - (y + uniform01(j.y)) * dy; // MainWindow.cpp:281-284
                r = generateRay(F.cam, sx, sy);
                L = v3(0, 0, 0); T = v3(1, 1, 1);
                depth = 0; sp = 0; block = 1;
                fresh = false;
            }
            const uint4 u = philoxBlock(pixel, (uint32_t)s, block++, F.seed); // this ray's draws, by slot
            bool alive = false; // does the current path continue with (r, T, depth)?
            rays++;
            Hit h;
            if (sceneIntersect<MESH>(S, r, h, pr))
            {
                const rtb_material &m = smat[h.mat];
                const V3 n = h.n;
                const V3 nl = (dot(n, r.d) < 0) ? n : n * -1;
                V3 local = matLocal(m, r, h.pos, n);
                const V3 emission = matEmission(m, h.pos);
                const float maxColor = (local.x + local.y + local.z) * 0.333333f;
                bool stop = false;
                if (++depth > F.setting.max_depth) stop = true;
                if (!stop && depth > F.setting.termination_depth)
                {
                    if (uniform01(u.x) < maxColor) local = local * (1 / maxColor);
                    else stop = true;
                }
                if (!stop && depth > RTB_MAX_DEPTH) stop = true;
                if (stop) L = L + mul(T, emission);
                else
                {
                    const float p_type = uniform01(u.y);
                    const float dif = m.diffusiveness, ref = m.reflectiveness, rfr = m.refractiveness;
                    if (dif > 0 && p_type < dif)
                    { // uniform hemisphere about nl, unit weight (MainWindow.cpp:185-200)
                        const float r1 = uniform01(u.z), r2 = uniform01(u.w);
                        const float theta = 2 * PI_F * r1;
#if RTB_MC_REFERENCE_TRIG
                        const float phi = acosf(r2);
                        const float ct = cosf(theta), st = sinf(theta), cp = cosf(phi), sn = sinf(phi);
#else
                        // cos(acos(r2)) = r2 and sin(acos(r2)) = sqrt(1 - r2^2): the same direction to float rounding (the reference's
                        // libm calls and CUDA's differ in the last ulps anyway; Monte-Carlo parity is statistical, SURVEY 8c)
                        float st, ct;
                        sincosf(theta, &st, &ct);
                        const float cp = r2, sn = sqrtf(fmaxf(1.0f - r2 * r2, 0.0f));
#endif
                        const V3 w = nl;
                        const V3 uu = (fabsf(w.x) >= 0.1f) ? normalize(cross(v3(0, 1, 0), w)) : normalize(cross(v3(1, 0, 0), w));
                        const V3 v = cross(w, uu);
                        const V3 dir = uu * (ct * sn) + v * (st * sn) + w * cp;
                        L = L + mul(T, emission); T = mul(T, local);
                        r.o = h.pos; r.d = dir; alive = true;
                    }
                    else if (ref > 0 && p_type >= dif && p_type <= dif + ref)
                    {
                        L = L + mul(T, emission); T = mul(T, local);
                        const V3 v = r.d - nl * 2 * dot(nl, r.d);
                        r.o = h.pos; r.d = v; alive = true;
                    }
                    else if (rfr > 0 && p_type > dif + ref)
                    {
                        const Fresnel f = refraction(r, n, nl, m.refractive_index);
                        if (f.tir)
                        {
                            L = L + mul(T, emission); T = mul(T, local);
                            r.o = h.pos; r.d = f.refl; alive = true;
                        }
                        else if (depth > F.setting.single_tracing_depth)
                        {
                            if (uniform01(u.z) < f.P) { T = T * f.RP; r.d = f.refl; }
                            else { T = T * f.TP; r.d = f.tdir; }
                            r.o = h.pos; alive = true;
                        }
                        else
                        {
                            if (sp < RTB_MC_STACK)
                            {
                                stack[sp].o = h.pos; stack[sp].d = f.refl; stack[sp].T = T * f.Re; stack[sp].depth = depth; sp++;
                            }
                            T = T * f.Tr; r.o = h.pos; r.d = f.tdir; alive = true;
                        }
                    }
                    else L = L + mul(T, emission); // "impossible to reach" tail, MainWindow.cpp:247-248
                }
            }
            // one way round the loop for every lane (no `continue`: lanes that leave an iteration at different points would
            // otherwise run the next iterations apart -- measured 13.8 of 32 lanes per instruction with early continues)
            if (!alive)
            {
                if (sp > 0)
                {
                    --sp;
                    r.o = stack[sp].o; r.d = stack[sp].d; T = stack[sp].T; depth = stack[sp].depth;
                }
                else
                {
                    acc = acc + L * inv; // MainWindow.cpp:288
                    if (F.moments) { sum = sum + L; sumsq = sumsq + mul(L, L); }
                    s++;
                    fresh = true;
                }
            }
        }
        if (F.moments)
        {
            float *o = out + 6 * pixelSlot(F, x, lr, y);
            o[0] = sum.x; o[1] = sum.y; o[2] = sum.z; o[3] = sumsq.x; o[4] = sumsq.y; o[5] = sumsq.z;
        }
        else storeColor(F, out, x, lr, y, acc);
    }
    finishWarp(F, counters, tile, t_start, rays, ProbeCounts<Probe>::tris(pr), ProbeCounts<Probe>::steps(pr));
}

} // namespace rtb
