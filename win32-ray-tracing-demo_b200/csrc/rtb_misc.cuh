// rtb_misc.cuh -- the non-template kernels of the library (sm_100a): tile-order counting sort, parity hooks
// (primary rays with traversal recording, ray batches), ray, closest-point, winding-number and triangle queries, the PerformanceTest
// bounce loop, frame un-sharding.
// Included by exactly one translation unit (rtb_abi.cu).
#pragma once
#include "rtb_kernels.cuh"
#include "rtb_closest.h"
#include "rtb_winding.h"
#include "rtb_tritri.h"

namespace rtb {

// ---- heaviest-first tile order from the recorded costs: a counting sort over 128 log-scale buckets ----
__device__ __forceinline__ int costBucket(unsigned int c)
{ // 4 buckets per power of two, bucket 127 = heaviest
    if (c < 4) return (int)c;
    const int e = 31 - __clz(c);
    return e * 4 + (int)((c >> (e - 2)) & 3u) - 4;
}

// Sorting unit u: tile u, or -- group mode (FrameParams::group4) -- four adjacent tiles which one CTA renders together: it is
// busy for as long as its slowest tile, so that is the group's cost.  Groups count as four tiles in the histogram and take four
// consecutive entries of the order; all offsets stay in tiles.  group 1: tiles 4u .. 4u + 3 of a tile row; group 2: tiles
// (4 gy + k) * tiles_x + tx, k = 0 .. 3, of a tile column (u = gy * tiles_x + tx).
__device__ __forceinline__ uint4 unitTiles(int u, int group, int tiles_x)
{
    if (group == 2)
    {
        const int gy = u / tiles_x, tx = u - gy * tiles_x;
        const unsigned int t = (unsigned int)(4 * gy * tiles_x + tx), sx = (unsigned int)tiles_x;
        return make_uint4(t, t + sx, t + 2u * sx, t + 3u * sx);
    }
    return make_uint4(4u * u, 4u * u + 1u, 4u * u + 2u, 4u * u + 3u);
}
__device__ __forceinline__ unsigned int unitCost(const unsigned int *__restrict__ cost, int u, int group, int tiles_x)
{
    if (!group) return cost[u];
    const uint4 t = unitTiles(u, group, tiles_x);
    return max(max(cost[t.x], cost[t.y]), max(cost[t.z], cost[t.w]));
}

__global__ void k_cost_histogram(const unsigned int *__restrict__ cost, int n, unsigned int *__restrict__ hist, int group, int tiles_x)
{
    __shared__ unsigned int h[RTB_COST_BUCKETS];
    for (int i = threadIdx.x; i < RTB_COST_BUCKETS; i += blockDim.x) h[i] = 0;
    __syncthreads();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) atomicAdd(&h[costBucket(unitCost(cost, i, group, tiles_x))], group ? 4u : 1u);
    __syncthreads();
    for (int i = threadIdx.x; i < RTB_COST_BUCKETS; i += blockDim.x)
        if (h[i]) atomicAdd(&hist[i], h[i]);
}

// one thread: hist[] -> descending exclusive offsets in cursor[], hist[] cleared for the next frame.
// Also sizes the two latency-critical sets at the head of the order:
//   (host)      the `wide_count` heaviest tiles: one warp per PIXEL with warp-parallel leaf tests
//               (rtb_chain_wide.cuh).  Their recorded costs are scaled up generously (FrameParams::cost_scale),
//               so a tile that is in the set stays in it until it really becomes light;
//   n_heavy[0]  those plus the tiles within `heavy_buckets` quarter-octaves of the heaviest tile that is NOT in
//               the first set, at most heavy_limit of them: resumable
//               traversal (rtb_chain_sm.cuh).
// n_heavy[1] = FLOOR BUCKET of the order: every tile in a bucket at or below it is "light" and is placed in one
// common bucket, i.e. (nearly) in raster order instead of by cost.  With floor_delta > 0 the floor lies that many
// quarter-octaves above the median tile (9: tiles up to ~4.8x the median are light).  Heaviest-first only matters
// for the tiles that can stretch the end of the kernel; among the light ones raster order keeps neighbouring tiles
// -- neighbouring framebuffer rows -- in flight together.  When the kernels store straight into the caller's
// page-locked host frame that is what lets the 96-byte row segments of adjacent tiles combine into long PCIe
// writes: 4K SAH frame 6.95 -> 5.79 ms with the floor, against 5.48 ms into HBM (profiles/r01_e2e_floor_bucket.log).
// Frames rendered into device memory keep floor_delta = 0 (pure heaviest-first is 3 % faster there).
// heavy_alpha > 0 selects the latency-critical set by TIME instead of by distance from the heaviest tile: with every tile's
// recorded cost c (cycles it took in the throughput kernel, on a saturated SM) the kernel's balanced finishing time is about
// T* = sum(c) / resident warp slots; a tile whose own c exceeds heavy_alpha * T* would still be running when everything else
// is done, wherever it is started -- those go to the latency tier (at most heavy_limit of them).  Unlike "within 2x of the
// heaviest tile" this does not shrink the set of a shard that happens to hold one outlier tile.
__global__ void k_cost_offsets(unsigned int *__restrict__ hist, unsigned int *__restrict__ cursor, unsigned int *__restrict__ n_heavy,
                               int n_tiles, int heavy_buckets, int heavy_limit, int wide_count, int floor_delta, float heavy_alpha,
                               int warp_slots)
{
    // launched with RTB_COST_BUCKETS threads: the histogram is fetched (and cleared for the next frame) in parallel,
    // the short serial pass below then runs out of shared memory (18 -> ~4 us; it sits at the end of every frame)
    __shared__ unsigned int h[RTB_COST_BUCKETS];
    for (int b = threadIdx.x; b < RTB_COST_BUCKETS; b += blockDim.x) { h[b] = hist[b]; hist[b] = 0; }
    __syncthreads();
    if (threadIdx.x == 0)
    {
        int floorBucket = 0;
        if (floor_delta > 0)
        {
            unsigned int below = 0;
            int median = 0;
            for (int b = 0; b < RTB_COST_BUCKETS; b++)
            {
                below += h[b];
                if (2u * below >= (unsigned int)n_tiles) { median = b; break; }
            }
            floorBucket = min(median + floor_delta, RTB_COST_BUCKETS - 1);
        }
        const unsigned int wide = (unsigned int)min(wide_count, n_tiles);
        unsigned int run = 0, heavy = wide;
        int top2 = -1; // bucket of the heaviest tile outside the wide set
        for (int b = RTB_COST_BUCKETS - 1; b >= 0; b--)
        {
            if (b >= floorBucket) cursor[b] = run; // buckets below the floor are placed through cursor[floorBucket]
            run += h[b];
            if (top2 < 0 && run > wide) top2 = b;
            if (top2 >= 0 && b >= top2 - heavy_buckets) heavy = run;
        }
        if (heavy_alpha > 0.f)
        {
            // centre of bucket b (costBucket: 4 buckets per power of two): 2^e * (1 + (q + 0.5) / 4), e = (b + 4) / 4, q = (b + 4) % 4
            double total = 0;
            for (int b = 4; b < RTB_COST_BUCKETS; b++) total += (double)h[b] * ldexp(1.0 + (((b + 4) & 3) + 0.5) * 0.25, (b + 4) >> 2);
            const double limit = (double)heavy_alpha * total / (double)max(warp_slots, 1);
            unsigned int r2 = 0;
            heavy = wide;
            for (int b = RTB_COST_BUCKETS - 1; b >= 4; b--)
            {
                if (ldexp(1.0 + (((b + 4) & 3) + 0.5) * 0.25, (b + 4) >> 2) < limit) break;
                r2 += h[b];
                heavy = max(heavy, r2);
            }
        }
        if (heavy < wide) heavy = wide;
        // a bucket may be cut: with whole buckets only, a well-filled bucket at the top (flat cost distributions)
        // would leave no latency-critical set at all
        if (heavy - wide > (unsigned int)heavy_limit) heavy = wide + (unsigned int)heavy_limit;
        n_heavy[0] = heavy;
        n_heavy[1] = (unsigned int)floorBucket;
    }
}

// Each block owns a contiguous chunk of tiles: count per bucket in shared memory, reserve the chunk's
// range of every bucket with ONE global atomic per bucket, then place the tiles with shared-memory
// atomics (the naive per-tile global atomic took 146 us on the 345,600 tiles of a 4K frame).
__global__ void k_cost_scatter(const unsigned int *__restrict__ cost, int n, unsigned int *__restrict__ cursor,
                               unsigned int *__restrict__ order, const unsigned int *__restrict__ n_heavy, int group, int tiles_x)
{
    const unsigned int span = group ? 4u : 1u;
    const int floor_bucket = (int)n_heavy[1]; // written by k_cost_offsets just before this launch
    __shared__ unsigned int cnt[RTB_COST_BUCKETS], base[RTB_COST_BUCKETS];
    const int per = (n + gridDim.x - 1) / gridDim.x;
    const int begin = blockIdx.x * per, end = min(begin + per, n);
    for (int i = threadIdx.x; i < RTB_COST_BUCKETS; i += blockDim.x) cnt[i] = 0;
    __syncthreads();
    for (int i = begin + threadIdx.x; i < end; i += blockDim.x) atomicAdd(&cnt[max(costBucket(unitCost(cost, i, group, tiles_x)), floor_bucket)], span);
    __syncthreads();
    for (int i = threadIdx.x; i < RTB_COST_BUCKETS; i += blockDim.x)
    {
        base[i] = cnt[i] ? atomicAdd(&cursor[i], cnt[i]) : 0u;
        cnt[i] = 0;
    }
    __syncthreads();
    for (int i = begin + threadIdx.x; i < end; i += blockDim.x)
    {
        const int b = max(costBucket(unitCost(cost, i, group, tiles_x)), floor_bucket);
        const unsigned int at = base[b] + atomicAdd(&cnt[b], span);
        if (group) reinterpret_cast<uint4 *>(order)[at >> 2] = unitTiles(i, group, tiles_x); // `at` is a multiple of 4
        else order[at] = (unsigned int)i;
    }
}

// ---- k-d leaf lists on even positions of the reference array (upload time) --------------------------------------------------
// The list scans test two list positions per iteration out of the pair stream (pre2[p] = positions 2p, 2p + 1); a list that
// starts on an odd position costs half an iteration more on average -- one of the ~17 pair iterations per ray on the SAH tree.
// A leaf carries its own count, so the array can simply be re-laid out with every list on an even position: the slot behind an
// odd-length list is padding that lies outside every [first, first + count) and is never tested.  size[i] = padded length of
// leaf i (inner nodes 0); first = exclusive scan; the caller's layout is kept for rtb_scene_kd_download.
__global__ void k_kd_pad_sizes(const uint2 *__restrict__ nodes, int n, unsigned int *__restrict__ size)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    unsigned int v = 0;
    if (i < n)
    {
        const uint2 nd = nodes[i];
        if ((nd.y & 3u) == 3u) v = ((nd.y >> 2) + 1u) & ~1u;
    }
    size[i] = v; // size[n] = 0: the total of the scan lands in first[n]
}

__global__ void k_kd_relayout(const uint2 *__restrict__ nodes, int n, const unsigned int *__restrict__ first, const uint32_t *__restrict__ refs,
                              uint2 *__restrict__ nodes_out, uint32_t *__restrict__ refs_out, unsigned int cap)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint2 nd = nodes[i];
    if ((nd.y & 3u) == 3u)
    {
        const unsigned int count = nd.y >> 2, from = nd.x, to = first[i];
        if ((unsigned long long)to + ((count + 1u) & ~1u) <= cap) // (the capacity is the exact total: always true)
        {
            for (unsigned int j = 0; j < count; j++) refs_out[to + j] = refs[from + j];
            if (count & 1u) refs_out[to + count] = refs[from + count - 1u]; // padding: any valid index
            nd.x = to;
        }
        else nd.y = 3u; // never reached; an empty leaf rather than a list outside the array
    }
    nodes_out[i] = nd;
}

// ---------------------------------------------------------------------------------------------
// Parity hooks: primary rays with traversal recording, and arbitrary ray batches
// ---------------------------------------------------------------------------------------------
template <bool MESH = false>
__global__ void __launch_bounds__(RTB_CTA_THREADS)
k_trace_primary(const __grid_constant__ DScene S, const __grid_constant__ FrameParams F, int *__restrict__ hit_id,
                float *__restrict__ hit_t, int *__restrict__ seq_len, unsigned long long *__restrict__ seq_hash,
                int *__restrict__ seq_buf, int seq_cap)
{
    int x, lr, y;
    unsigned int tile;
    if (!pixelOfThread(F, x, lr, y, tile)) return;
    const float dx = 1.0f / F.height, dy = 1.0f / F.height;
    const float sx = (x + 0.5f) * dx, sy = 1 - (y + 0.5f) * dy;
    const Ray r = generateRay(F.cam, sx, sy);
    const size_t p = (size_t)y * F.width + x;
    SeqProbe pr;
    pr.buf = seq_buf ? seq_buf + p * seq_cap : nullptr;
    pr.cap = seq_buf ? seq_cap : 0;
    Hit h;
    const bool ok = sceneIntersect<MESH>(S, r, h, pr);
    if (hit_id) hit_id[p] = ok ? h.id : -1;
    if (hit_t) hit_t[p] = ok ? h.t : -1.0f;
    if (seq_len) seq_len[p] = pr.len;
    if (seq_hash) seq_hash[p] = pr.hash;
    if (seq_buf)
        for (int i = pr.len; i < seq_cap; i++) seq_buf[p * seq_cap + i] = -1;
}

// Ray queries (rtb_query_rays, rtb_intersect_rays): one lane per ray, the ray [6] floats read as three 64-bit loads.  The
// search starts at the ray's bound (rtb.h: a strict bound; at or above FLT_MAX it starts at FLT_MAX, as the unbounded search
// does -- +inf would accept hits at an infinite distance the unbounded search rejects; NaN or <= 0.0005 is a miss, every
// accepted t being >= 0.0005).  ANY: occluded[i] = 1 exactly when the closest query with the same bound hits.
struct QueryParams
{
    long long n;
    const float *rays, *tmax; // tmax: [n] per-ray bounds, or null: tmax_all for every ray
    float tmax_all;
    int *hit_id;
    float *hit_t, *position, *normal;
    uint8_t *occluded;
};

template <bool MESH, bool ANY>
__global__ void __launch_bounds__(RTB_CTA_THREADS)
k_query_rays(const __grid_constant__ DScene S, const __grid_constant__ QueryParams Q)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Q.n) return;
    const float2 *rp = reinterpret_cast<const float2 *>(Q.rays) + 3 * i;
    const float2 a = __ldg(rp), b = __ldg(rp + 1), c = __ldg(rp + 2);
    Ray r;
    r.o = v3(a.x, a.y, b.x);
    r.d = v3(b.y, c.x, c.y);
    const float bound = Q.tmax ? __ldg(Q.tmax + i) : Q.tmax_all;
    NoProbe pr;
    Hit h;
    const bool ok = bound > 0.0005f && sceneIntersect<MESH, ANY>(S, r, h, pr, fminf(bound, FLT_MAX));
    if (ANY)
    {
        Q.occluded[i] = ok ? 1 : 0;
        return;
    }
    if (Q.hit_id) Q.hit_id[i] = ok ? h.id : -1;
    if (Q.hit_t) Q.hit_t[i] = ok ? h.t : -1.0f;
    if (Q.position) { Q.position[3 * i] = ok ? h.pos.x : 0; Q.position[3 * i + 1] = ok ? h.pos.y : 0; Q.position[3 * i + 2] = ok ? h.pos.z : 0; }
    if (Q.normal) { Q.normal[3 * i] = ok ? h.n.x : 0; Q.normal[3 * i + 1] = ok ? h.n.y : 0; Q.normal[3 * i + 2] = ok ? h.n.z : 0; }
}

// Point queries (rtb_query_points): the nearest point on the TRIANGLES and MESH records within a strict per-point radius
// (include/rtb.h, DESIGN 3e).  Distances are rtb_closest.h's squared distances d2; a pair is accepted when d2 < best, best
// starting at fl(r * r).
struct PointParams
{
    long long n;
    const float *points, *rmax; // rmax: [n] per-point radii, or null: rmax_all for every point
    float rmax_all;
    int *hit_id;
    float *distance, *position, *normal;
    uint8_t *near;
};

__device__ __forceinline__ float closestOf(const float4 *tris, unsigned int idx, const float p[3])
{
    const TriData T = loadTri(tris, idx);
    const float t[9] = {T.q0.x, T.q0.y, T.q0.z, T.q0.w, T.q1.x, T.q1.y, T.q1.z, T.q1.w, T.q2.x};
    float q[3];
    return rtb_closest::closestPoint(p, t, q);
}

// The hierarchy of a MESH record, walked from the root: both children's box distances per step, the nearer child first, the
// other pushed with its distance and dropped when popped above the current best.  Nearest (d2, k) in lexicographic order;
// `best` comes in as the earlier records' nearest d2 (or the bound) and bestK as -1, so the mesh replaces it only with a
// strictly smaller d2, as the run's `d2 < best` does.  A node with boxDist2 > best holds no winner (rtb_closest.h), so the
// result is the run's whatever the tree's shape.  ANY: ends at the first accepted triangle.  Returns the leaf position won.
template <bool ANY>
__device__ int meshClosest(const DScene &S, unsigned int base, const float p[3], float &best, int &bestK)
{
    const float4 *nodes = S.mesh_nodes + 4ull * base;
    int stackNode[RTB_BVH_STACK];
    float stackDist[RTB_BVH_STACK];
    int sp = 0, node = 0, won = -1;
    auto leaf = [&](int pos) {
        const float d2 = closestOf(S.mesh_tris, base + (unsigned int)pos, p);
        if (!(d2 <= best)) return;
        const int k = (int)__ldg(S.mesh_order + base + pos);
        if (d2 < best || k < bestK) { best = d2; bestK = k; won = pos; }
    };
    while (true)
    {
        const float4 *q = nodes + 4ull * (unsigned int)node;
        const float4 q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2), q3 = __ldg(q + 3);
        const float lo0[3] = {q0.x, q0.y, q0.z}, lo1[3] = {q0.w, q1.x, q1.y};
        const float hi0[3] = {q1.z, q1.w, q2.x}, hi1[3] = {q2.y, q2.z, q2.w};
        const int c0 = __float_as_int(q3.x), c1 = __float_as_int(q3.y);
        const float b0 = rtb_closest::boxDist2(p, lo0, hi0);
        const bool two = c1 != c0; // a one-triangle mesh links its leaf twice
        const float b1 = two ? rtb_closest::boxDist2(p, lo1, hi1) : INFINITY;
        if (c0 < 0 && b0 <= best) leaf(~c0);
        if (two && c1 < 0 && b1 <= best) leaf(~c1);
        if (ANY && won >= 0) break;
        const bool in0 = c0 >= 0 && b0 <= best, in1 = c1 >= 0 && b1 <= best;
        if (in0 && in1)
        {
            const bool first1 = b1 < b0;
            stackNode[sp] = first1 ? c0 : c1;
            stackDist[sp++] = first1 ? b0 : b1;
            node = first1 ? c1 : c0;
        }
        else if (in0) node = c0;
        else if (in1) node = c1;
        else
        {
            while (sp > 0 && stackDist[sp - 1] > best) sp--;
            if (sp == 0) break;
            node = stackNode[--sp];
        }
    }
    return won;
}

template <bool ANY>
__global__ void __launch_bounds__(RTB_CTA_THREADS)
k_query_points(const __grid_constant__ DScene S, const __grid_constant__ PointParams Q)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Q.n) return;
    const float p[3] = {__ldg(Q.points + 3 * i), __ldg(Q.points + 3 * i + 1), __ldg(Q.points + 3 * i + 2)};
    const float r = Q.rmax ? __ldg(Q.rmax + i) : Q.rmax_all;
    float best = r * r;
    int id = -1;
    const float4 *winner = nullptr; // the winning triangle's record
    if (r > 0.0f && p[0] == p[0] && p[1] == p[1] && p[2] == p[2]) // NaN or r <= 0: a miss without a walk
        for (int j = 0; j < S.n_prims; j++)
        {
            const rtb_prim &P = S.prims[j];
            if (ANY && id >= 0) break;
            if (P.type == RTB_PRIM_TRIANGLES)
            {
                for (int k = 0; k < P.count; k++)
                {
                    const float d2 = closestOf(S.loose, (unsigned int)(P.first + k), p);
                    if (d2 < best)
                    {
                        best = d2; id = P.base_id + k; winner = S.loose + 3ull * (unsigned int)(P.first + k);
                        if (ANY) break;
                    }
                }
            }
            else if (P.type == RTB_PRIM_MESH)
            {
                int k = -1;
                const int pos = meshClosest<ANY>(S, (unsigned int)S.mesh_base[j], p, best, k);
                if (pos >= 0) { id = P.base_id + k; winner = S.mesh_tris + 3ull * ((unsigned int)S.mesh_base[j] + (unsigned int)pos); }
            }
        }
    if (ANY)
    {
        Q.near[i] = id >= 0 ? 1 : 0;
        return;
    }
    float q[3] = {0.0f, 0.0f, 0.0f}, nrm[3] = {0.0f, 0.0f, 0.0f};
    if (id >= 0)
    { // the winner's closest point again: the same function on the same record, so the same bits as in the search
        const TriData T = loadTri(winner, 0);
        const float t[9] = {T.q0.x, T.q0.y, T.q0.z, T.q0.w, T.q1.x, T.q1.y, T.q1.z, T.q1.w, T.q2.x};
        rtb_closest::closestPoint(p, t, q);
        nrm[0] = T.q2.y; nrm[1] = T.q2.z; nrm[2] = T.q2.w;
    }
    if (Q.hit_id) Q.hit_id[i] = id;
    if (Q.distance) Q.distance[i] = id >= 0 ? sqrtf(best) : -1.0f;
    if (Q.position) { Q.position[3 * i] = q[0]; Q.position[3 * i + 1] = q[1]; Q.position[3 * i + 2] = q[2]; }
    if (Q.normal) { Q.normal[3 * i] = nrm[0]; Q.normal[3 * i + 1] = nrm[1]; Q.normal[3 * i + 2] = nrm[2]; }
}

// Winding-number queries (rtb_query_winding): w(p) = sum of the TRIANGLES and MESH records' solid angles / 4 pi (include/rtb.h,
// DESIGN 3f).  The moments are rtb_scene's, not DScene's, so no other kernel's parameters change.
struct WindingParams
{
    long long n;
    const float *points;
    const float4 *moments; // rtb_scene::mesh_moments: 4 float4 per node slot, parallel to DScene::mesh_nodes
    float beta;
    float *winding;
    uint8_t *inside;
};

// one triangle's exact term, fl(Omega * fl(1 / 4 pi))
__device__ __forceinline__ float windingOf(const float4 *tris, unsigned int idx, const float p[3])
{
    const TriData T = loadTri(tris, idx);
    const float t[9] = {T.q0.x, T.q0.y, T.q0.z, T.q0.w, T.q1.x, T.q1.y, T.q1.z, T.q1.w, T.q2.x};
    return rtb_winding::solidAngle(p, t) * RTB_WINDING_INV4PI;
}

// The hierarchy of a MESH record, walked from the root with nothing pruned: per step the child links and both children's
// moments {N0, c0, r0, N1, c1, r1}; a leaf child adds its exact term, an inner child farther than beta r adds its dipole,
// any other child is descended into (the first, the second pushed).  w comes in as the earlier records' sum.
__device__ float meshWinding(const DScene &S, const float4 *moments, unsigned int base, const float p[3], float beta, float w)
{
    const float4 *nodes = S.mesh_nodes + 4ull * base, *mom = moments + 4ull * base;
    int stack[RTB_BVH_STACK];
    int sp = 0, node = 0;
    while (true)
    {
        const float4 q3 = __ldg(nodes + 4ull * (unsigned int)node + 3);
        const float4 *m = mom + 4ull * (unsigned int)node;
        const float4 m0 = __ldg(m), m1 = __ldg(m + 1), m2 = __ldg(m + 2), m3 = __ldg(m + 3);
        const int ch[2] = {__float_as_int(q3.x), __float_as_int(q3.y)};
        const float N[2][3] = {{m0.x, m0.y, m0.z}, {m1.w, m2.x, m2.y}};
        const float c[2][3] = {{m0.w, m1.x, m1.y}, {m2.z, m2.w, m3.x}};
        const float r[2] = {m1.z, m3.y};
        const int sides = ch[1] != ch[0] ? 2 : 1; // a one-triangle mesh links its leaf twice
        bool down[2] = {false, false};
        for (int s = 0; s < sides; s++)
        {
            if (ch[s] < 0) w += windingOf(S.mesh_tris, base + (unsigned int)~ch[s], p);
            else if (rtb_winding::far(p, c[s], r[s], beta)) w += rtb_winding::dipole(p, N[s], c[s]);
            else down[s] = true;
        }
        if (down[0] && down[1])
        {
            stack[sp++] = ch[1];
            node = ch[0];
        }
        else if (down[0]) node = ch[0];
        else if (down[1]) node = ch[1];
        else
        {
            if (sp == 0) break;
            node = stack[--sp];
        }
    }
    return w;
}

__global__ void __launch_bounds__(RTB_CTA_THREADS)
k_query_winding(const __grid_constant__ DScene S, const __grid_constant__ WindingParams Q)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Q.n) return;
    const float p[3] = {__ldg(Q.points + 3 * i), __ldg(Q.points + 3 * i + 1), __ldg(Q.points + 3 * i + 2)};
    float w = 0.0f;
    if (!(p[0] == p[0] && p[1] == p[1] && p[2] == p[2])) w = NAN; // a NaN point: NaN / outside, without a walk
    else
        for (int j = 0; j < S.n_prims; j++)
        {
            const rtb_prim &P = S.prims[j];
            if (P.type == RTB_PRIM_TRIANGLES)
                for (int k = 0; k < P.count; k++) w += windingOf(S.loose, (unsigned int)(P.first + k), p);
            else if (P.type == RTB_PRIM_MESH)
                w = meshWinding(S, Q.moments, (unsigned int)S.mesh_base[j], p, Q.beta, w);
        }
    if (Q.winding) Q.winding[i] = w;
    if (Q.inside) Q.inside[i] = w > 0.5f ? 1 : 0;
}

// Triangle queries (rtb_query_triangles): which TRIANGLES and MESH triangles each query triangle shares a point with, decided
// exactly by rtb_tritri.h (include/rtb.h, DESIGN 3g).  ANY: hit[i]; otherwise every pair (i, hit_id) is counted in *count and
// stored while the count is below capacity.
struct TriQueryParams
{
    long long n;
    const float *tris; // [n][12] a, b, c, normal; 16-byte aligned
    uint8_t *hit;
    int2 *pairs;
    long long capacity;
    unsigned long long *count;
};

// One pair, appended with one atomic per group of lanes that report together.
__device__ __forceinline__ void appendPair(const TriQueryParams &Q, int i, int id)
{
    const unsigned int mask = __activemask();
    const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
    unsigned long long at = 0;
    if (lane == leader) at = atomicAdd(Q.count, (unsigned long long)__popc(mask));
    at = __shfl_sync(mask, at, leader) + (unsigned long long)__popc(mask & ((1u << lane) - 1u));
    if (at < (unsigned long long)Q.capacity) Q.pairs[at] = make_int2(i, id);
}

// the scene triangle at packed position idx as (a, fl(a - e1), fl(a - e2)), and whether it meets the query triangle p
__device__ __forceinline__ bool triMeets(const float4 *tris, unsigned int idx, const float p[9], const float lo[3], const float hi[3])
{
    const TriData T = loadTri(tris, idx);
    const float t[9] = {T.q0.x, T.q0.y, T.q0.z, T.q0.x - T.q0.w, T.q0.y - T.q1.x, T.q0.z - T.q1.y,
                        T.q0.x - T.q1.z, T.q0.y - T.q1.w, T.q0.z - T.q2.x};
    float tlo[3], thi[3];
    rtb_tritri::box(t, tlo, thi);
    return rtb_tritri::boxesOverlap(lo, hi, tlo, thi) && rtb_tritri::meets(p, t);
}

// The hierarchy of a MESH record, walked from the root with meshClosest's node loads: both children's boxes per step against
// the query triangle's box, an overlapping leaf tested, overlapping inner children descended (the first, the second pushed).
// ANY: returns true at the first pair.
template <bool ANY>
__device__ bool meshTriangles(const DScene &S, const TriQueryParams &Q, unsigned int base, int baseId, int i, const float p[9],
                              const float lo[3], const float hi[3])
{
    const float4 *nodes = S.mesh_nodes + 4ull * base;
    int stack[RTB_BVH_STACK];
    int sp = 0, node = 0;
    while (true)
    {
        const float4 *q = nodes + 4ull * (unsigned int)node;
        const float4 q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2), q3 = __ldg(q + 3);
        const float lo0[3] = {q0.x, q0.y, q0.z}, lo1[3] = {q0.w, q1.x, q1.y};
        const float hi0[3] = {q1.z, q1.w, q2.x}, hi1[3] = {q2.y, q2.z, q2.w};
        const int c[2] = {__float_as_int(q3.x), __float_as_int(q3.y)};
        const int sides = c[1] != c[0] ? 2 : 1; // a one-triangle mesh links its leaf twice
        const bool o[2] = {rtb_tritri::boxesOverlap(lo, hi, lo0, hi0), sides == 2 && rtb_tritri::boxesOverlap(lo, hi, lo1, hi1)};
        for (int s = 0; s < sides; s++)
            if (c[s] < 0 && o[s] && triMeets(S.mesh_tris, base + (unsigned int)~c[s], p, lo, hi))
            {
                if (ANY) return true;
                appendPair(Q, i, baseId + (int)__ldg(S.mesh_order + base + (unsigned int)~c[s]));
            }
        const bool in0 = c[0] >= 0 && o[0], in1 = c[1] >= 0 && o[1];
        if (in0 && in1)
        {
            stack[sp++] = c[1];
            node = c[0];
        }
        else if (in0) node = c[0];
        else if (in1) node = c[1];
        else
        {
            if (sp == 0) break;
            node = stack[--sp];
        }
    }
    return false;
}

template <bool ANY>
__global__ void __launch_bounds__(RTB_CTA_THREADS)
k_query_triangles(const __grid_constant__ DScene S, const __grid_constant__ TriQueryParams Q)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Q.n) return;
    const float4 *t4 = reinterpret_cast<const float4 *>(Q.tris) + 3 * i;
    const float4 a = __ldg(t4), b = __ldg(t4 + 1), c = __ldg(t4 + 2);
    const float p[9] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x};
    bool found = false;
    if (!rtb_tritri::degenerate(p))
    {
        float lo[3], hi[3];
        rtb_tritri::box(p, lo, hi);
        for (int j = 0; j < S.n_prims && !(ANY && found); j++)
        {
            const rtb_prim &P = S.prims[j];
            if (P.type == RTB_PRIM_TRIANGLES)
            {
                for (int k = 0; k < P.count; k++)
                    if (triMeets(S.loose, (unsigned int)(P.first + k), p, lo, hi))
                    {
                        found = true;
                        if (ANY) break;
                        appendPair(Q, (int)i, P.base_id + k);
                    }
            }
            else if (P.type == RTB_PRIM_MESH)
                found = meshTriangles<ANY>(S, Q, (unsigned int)S.mesh_base[j], P.base_id, (int)i, p, lo, hi) || found;
        }
    }
    if (ANY) Q.hit[i] = found ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------
// PerformanceTest workload (reference src/PerformanceTest/main.cpp:29-59): mirror-reflect each ray until
// it hits a PLANE geometry (the plane closing the tunnel exit), misses, or exceeds max_depth.
// ---------------------------------------------------------------------------------------------
// WIDE = false: one lane per ray (batches that fill the device).  WIDE = true: one WARP per ray -- the 32 lanes walk the
// accelerator in lock step and test 32 triangles of a leaf / cell list at once (nearestInList<.., WIDE>), as in the
// warp-per-pixel render tier: the reference program's own batch is 1000 rays, which as 1000 threads occupies 8 CTAs and
// takes as long as its longest 200-bounce chain walked by one lane; as 1000 warps it fills the device.  Results are
// identical (same arithmetic; ties in a list go to the earliest position).  k-d trees and grids only.
template <bool WIDE, bool MESH = false>
__global__ void __launch_bounds__(RTB_CTA_THREADS)
k_bounce_rays(const __grid_constant__ DScene S, long long n, const float *__restrict__ rays, int max_depth,
              int *__restrict__ reached, int *__restrict__ depth_out, int *__restrict__ last_id, float *__restrict__ last_pos,
              unsigned long long *__restrict__ total_rays, unsigned long long *__restrict__ next_ray)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool writer = !WIDE || (threadIdx.x & 31) == 0;
    unsigned int traced = 0;
    // One lane per ray: the chains are 1 .. 200 bounces long (35 on average), so a lane that has finished its ray takes the
    // next one from a queue (`next_ray`, one atomic per ray) instead of idling until the longest chain of its warp ends.
    // The launch is sized to the device, not to the batch.  Rays are independent: the order changes no result.
    for (long long i = WIDE ? (t >> 5) : (long long)atomicAdd(next_ray, 1ull); i < n; i = WIDE ? n : (long long)atomicAdd(next_ray, 1ull))
    {
        Ray r;
        r.o = v3(rays[6 * i], rays[6 * i + 1], rays[6 * i + 2]);
        r.d = v3(rays[6 * i + 3], rays[6 * i + 4], rays[6 * i + 5]);
        NoProbe pr;
        int depth = 0, ok = 0, id = -1;
        V3 pos = v3(0, 0, 0);
        RayCtx ctx; // newRay.context = r.context, PerformanceTest/main.cpp:57
        ctx.inTunnel = 0; ctx.segment = -1;
        while (true)
        {
            Hit h;
            traced++;
            bool hit;
            if (WIDE)
                hit = sceneIntersectWith(S, r, h, pr, [&](int &tri, float &tt, V3 &nn) {
                    if (S.accel == RTB_ACCEL_REGULAR_GRID || S.accel == RTB_ACCEL_FLAT_GRID) return gridIntersect<true>(S, r, tri, tt, nn, pr);
                    return kdIntersect<true>(S, r, tri, tt, nn, pr);
                });
            else hit = sceneIntersect<MESH>(S, r, h, pr, ctx);
            if (!hit) { id = -1; break; }
            id = h.id; pos = h.pos;
            const V3 nl = (dot(h.n, r.d) < 0) ? h.n : h.n * -1;
            if (++depth > max_depth) break;
            if (h.prim_type == RTB_PRIM_PLANE) { ok = 1; break; }
            const V3 v = r.d - nl * 2 * dot(nl, r.d);
            r.o = h.pos;
            r.d = v;
        }
        if (writer)
        {
            if (reached) reached[i] = ok;
            if (depth_out) depth_out[i] = depth;
            if (last_id) last_id[i] = id;
            if (last_pos) { last_pos[3 * i] = pos.x; last_pos[3 * i + 1] = pos.y; last_pos[3 * i + 2] = pos.z; }
        }
    }
    if (!writer) traced = 0;
    traced = __reduce_add_sync(0xffffffffu, traced);
    if ((threadIdx.x & 31) == 0 && traced) atomicAdd(total_rays, (unsigned long long)traced);
}

// ---------------------------------------------------------------------------------------------
// Un-shard: after the NCCL all-gather the frame lives as [world][rows_per_rank][width][3] in
// block-cyclic row order; this puts it back into image row order [height][width][3].
// Pure 128-bit copies when width*3 floats is a multiple of 4 (every 4:3 frame is).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_unshard(const float *__restrict__ gathered, float *__restrict__ image, int width, int height, int world, int row_block,
          int rows_per_rank)
{
    const int y = blockIdx.y;
    const int b = y / row_block, rank = b % world, lb = b / world;
    const int lr = lb * row_block + (y - b * row_block);
    const size_t rowFloats = (size_t)width * 3;
    const float *src = gathered + ((size_t)rank * rows_per_rank + lr) * rowFloats;
    float *dst = image + (size_t)y * rowFloats;
    if ((rowFloats & 3) == 0)
    {
        const float4 *s4 = reinterpret_cast<const float4 *>(src);
        float4 *d4 = reinterpret_cast<float4 *>(dst);
        for (size_t i = blockIdx.x * blockDim.x + threadIdx.x; i < rowFloats / 4; i += (size_t)gridDim.x * blockDim.x) d4[i] = s4[i];
    }
    else
        for (size_t i = blockIdx.x * blockDim.x + threadIdx.x; i < rowFloats; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

// Column-block shards (localToGlobal): gathered = [world][height][width / world][3]; one thread per float4 of a
// column block row segment (col_block is a multiple of 8 pixels = 96 bytes)
__global__ void __launch_bounds__(256)
k_unshard_cols(const float *__restrict__ gathered, float *__restrict__ image, int width, int height, int world, int row_block,
               int col_block)
{
    const int y = blockIdx.y;
    const int by = y / row_block;
    const int localWidth = width / world;
    const int segFloat4 = col_block * 3 / 4, nbx = width / col_block;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nbx * segFloat4; i += gridDim.x * blockDim.x)
    {
        const int bx = i / segFloat4, q = i - bx * segFloat4;
        const int rank = (bx + by) % world;
        const int xl0 = (bx / world) * col_block;
        const float4 *src = reinterpret_cast<const float4 *>(gathered + (((size_t)rank * height + y) * localWidth + xl0) * 3);
        float4 *dst = reinterpret_cast<float4 *>(image + ((size_t)y * width + (size_t)bx * col_block) * 3);
        dst[q] = src[q];
    }
}

// A rank's local shard image -> its place in the whole frame (RTB_LAYOUT_GLOBAL addressing), as ONE streaming pass of
// 128-bit copies: the alternative to storing tile by tile into a peer-mapped frame while rendering (rtb_scatter_shard_device).
// One thread per float4; a local row is [local_width][3] floats; column-block shards move whole col_block segments.
__global__ void __launch_bounds__(256)
k_scatter_shard(const float *__restrict__ local, float *__restrict__ frame, int width, int height, int world, int rank, int row_block,
                int col_block, int local_width, int n_local_rows)
{
    const int lr = blockIdx.y;
    if (lr >= n_local_rows) return;
    int y;
    if (col_block) y = lr;
    else { const int lb = lr / row_block; y = (lb * world + rank) * row_block + (lr - lb * row_block); }
    if (y >= height) return;
    const int rowF4 = local_width * 3 / 4; // local_width % 4 == 0 (checked by the caller)
    const float4 *src = reinterpret_cast<const float4 *>(local + (size_t)lr * local_width * 3);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < rowF4; i += gridDim.x * blockDim.x)
    {
        int gx4 = i; // float4 index inside the frame row
        if (col_block)
        {
            const int segF4 = col_block * 3 / 4, c = i / segF4, q = i - c * segF4;
            int shift = (rank - y / row_block) % world;
            if (shift < 0) shift += world;
            gx4 = (c * world + shift) * segF4 + q;
        }
        reinterpret_cast<float4 *>(frame + (size_t)y * width * 3)[gx4] = src[i];
    }
}

} // namespace rtb
