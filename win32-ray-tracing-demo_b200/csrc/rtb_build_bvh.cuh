// rtb_build_bvh.cuh -- device build of the hierarchy of an RTB_PRIM_MESH record (include/rtb.h: rtb_bvhnode), from the raw
// loose-triangle records already on the device.  A linear BVH (Karras, "Maximizing parallelism in the construction of BVHs,
// octrees, and k-d trees", HPG 2012):
//   1. centroid bounds (float min / max through order-preserving integer atomics: exact, order-independent);
//   2. 62-bit keys: the 30-bit Morton code of the centroid, then the local index (32 bits) -- all keys differ, so every
//      inner node splits on a strictly lower bit than its parent and the depth of inner nodes is at most 62;
//   3. radix sort of the keys;
//   4. hierarchy: inner node i covers a key range found from the common-prefix lengths of its neighbours;
//   5. the local index of each leaf (the leaf order);
//   6. boxes bottom-up: the second thread to reach a node takes the union of its two child boxes (float min / max only);
//   7. the triangle records (exact stream) copied into leaf order.
// Every step is a deterministic function of the input: two builds of the same mesh are byte-identical.
// A refit (rtb_scene_mesh_update) keeps the child links and the leaf order: it derives the parent links from the child links
// (k_bvh_parents) and runs steps 6 and 7 again on the new records.
// Moments (k_bvh_moments, opt-in through rtb_scene_mesh_moments) follow step 7, after a build, a refit or a rebuild alike.
#pragma once
#include <cub/cub.cuh>
#include "rtb_bvh.h"
#include "rtb_winding.h"

namespace rtb {

__device__ __forceinline__ unsigned int orderedBits(float f)
{
    const unsigned int u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float orderedFloat(unsigned int u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u); }

__device__ __forceinline__ void triCentroid(const float *raw, unsigned int k, float c[3])
{
    const float *v = raw + 12ull * k;
    for (int i = 0; i < 3; i++) c[i] = (v[i] + v[3 + i] + v[6 + i]) * (1.0f / 3.0f);
}

// bounds[0..2] = ordered min, bounds[3..5] = ordered max of the centroids (initialised to 0xffffffff / 0)
__global__ void k_bvh_bounds(const float *__restrict__ raw, int n, unsigned int *__restrict__ bounds)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    float c[3];
    triCentroid(raw, (unsigned int)k, c);
    for (int i = 0; i < 3; i++)
    {
        atomicMin(bounds + i, orderedBits(c[i]));
        atomicMax(bounds + 3 + i, orderedBits(c[i]));
    }
}

__device__ __forceinline__ unsigned long long spread10(unsigned int v)
{
    unsigned long long x = v & 0x3ffu;
    x = (x | (x << 16)) & 0x030000FFull;
    x = (x | (x << 8)) & 0x0300F00Full;
    x = (x | (x << 4)) & 0x030C30C3ull;
    x = (x | (x << 2)) & 0x09249249ull;
    return x;
}

__global__ void k_bvh_keys(const float *__restrict__ raw, int n, const unsigned int *__restrict__ bounds, unsigned long long *__restrict__ keys)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    float c[3];
    triCentroid(raw, (unsigned int)k, c);
    unsigned long long m = 0;
    for (int i = 0; i < 3; i++)
    {
        const float lo = orderedFloat(bounds[i]), hi = orderedFloat(bounds[3 + i]);
        const float ext = hi - lo;
        float q = ext > 0.0f ? (c[i] - lo) / ext * 1024.0f : 0.0f;
        q = (q >= 0.0f) ? fminf(q, 1023.0f) : 0.0f; // NaN -> 0
        m |= spread10((unsigned int)q) << (2 - i);
    }
    keys[k] = (m << 32) | (unsigned int)k;
}

__device__ __forceinline__ int commonPrefix(const unsigned long long *keys, int n, int i, int j)
{
    if (j < 0 || j >= n) return -1;
    return __clzll(keys[i] ^ keys[j]);
}

// inner node i of n - 1 (n >= 2); parent links: 2 * parent + side, for inner nodes and leaves
__global__ void k_bvh_hierarchy(const unsigned long long *__restrict__ keys, int n, rtb_bvhnode *__restrict__ nodes,
                                int *__restrict__ parent_inner, int *__restrict__ parent_leaf)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const int d = (commonPrefix(keys, n, i, i + 1) - commonPrefix(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    const int dmin = commonPrefix(keys, n, i, i - d);
    int lmax = 2;
    while (commonPrefix(keys, n, i, i + lmax * d) > dmin) lmax *= 2;
    int l = 0;
    for (int t = lmax / 2; t >= 1; t /= 2)
        if (commonPrefix(keys, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = commonPrefix(keys, n, i, j);
    int s = 0, t = l;
    do
    {
        t = (t + 1) >> 1;
        if (commonPrefix(keys, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    const int split = i + s * d + (d < 0 ? -1 : 0);
    const int first = i < j ? i : j, last = i < j ? j : i;
    const int left = (first == split) ? ~split : split;
    const int right = (last == split + 1) ? ~(split + 1) : split + 1;
    nodes[i].child[0] = left;
    nodes[i].child[1] = right;
    nodes[i].pad_[0] = nodes[i].pad_[1] = 0;
    if (left < 0) parent_leaf[~left] = 2 * i; else parent_inner[left] = 2 * i;
    if (right < 0) parent_leaf[~right] = 2 * i + 1; else parent_inner[right] = 2 * i + 1;
}

// the parent links of a built hierarchy (the layout k_bvh_hierarchy writes), from its child links: inner node i of n - 1
__global__ void k_bvh_parents(const rtb_bvhnode *__restrict__ nodes, int n, int *__restrict__ parent_inner, int *__restrict__ parent_leaf)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    for (int side = 0; side < 2; side++)
    {
        const int c = nodes[i].child[side];
        if (c < 0) parent_leaf[~c] = 2 * i + side; else parent_inner[c] = 2 * i + side;
    }
}

// the local index of the triangle at each leaf position: the low half of its sorted key
__global__ void k_bvh_order(const unsigned long long *__restrict__ keys, int n, uint32_t *__restrict__ leaf_order)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) leaf_order[p] = (uint32_t)(keys[p] & 0xffffffffull);
}

// one thread per leaf position p: leaf box into its parent's slot, then up while this thread is the second to arrive
__global__ void k_bvh_boxes(const float *__restrict__ raw, const uint32_t *__restrict__ leaf_order, int n,
                            rtb_bvhnode *__restrict__ nodes, const int *__restrict__ parent_inner,
                            const int *__restrict__ parent_leaf, unsigned int *__restrict__ arrivals)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    float lo[3], hi[3];
    rtb_bvh::leafBox(raw + 12ull * leaf_order[p], lo, hi);
    if (n == 1)
    { // a single leaf: both links of the root point at it
        for (int c = 0; c < 2; c++)
        {
            for (int a = 0; a < 3; a++) { nodes[0].lo[c][a] = lo[a]; nodes[0].hi[c][a] = hi[a]; }
            nodes[0].child[c] = ~0;
        }
        nodes[0].pad_[0] = nodes[0].pad_[1] = 0;
        return;
    }
    int slot = parent_leaf[p];
    while (true)
    {
        const int node = slot >> 1, side = slot & 1;
        for (int a = 0; a < 3; a++) { nodes[node].lo[side][a] = lo[a]; nodes[node].hi[side][a] = hi[a]; }
        __threadfence();
        if (atomicAdd(arrivals + node, 1u) == 0u) return; // the sibling is still on its way: it continues
        __threadfence();
        const float *q = reinterpret_cast<const float *>(nodes + node);
        for (int a = 0; a < 3; a++)
        {
            lo[a] = fminf(__ldcg(q + a), __ldcg(q + 3 + a));
            hi[a] = fmaxf(__ldcg(q + 6 + a), __ldcg(q + 9 + a));
        }
        if (node == 0) return;
        slot = parent_inner[node];
    }
}

// triangle records in leaf order
__global__ void k_bvh_leaves(const float4 *__restrict__ exact, const uint32_t *__restrict__ leaf_order, int n,
                             float4 *__restrict__ leaf_tris)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const unsigned int k = leaf_order[p];
    for (int j = 0; j < 3; j++) leaf_tris[3ull * p + j] = exact[3ull * k + j];
}

// First-order moments of the winding queries (rtb_scene_mesh_moments), 16 floats per node slot, parallel to the nodes:
// {N0, c0, r0, N1, c1, r1, 0, 0} -- per child the area vector, the area-weighted centre and a radius about it that holds
// every vertex below.  Bottom-up with the arrival scheme of k_bvh_boxes, from the leaf-order records of k_bvh_leaves; the
// second thread to reach a node combines its two slots in child order, so the result does not depend on the arrival order.
__global__ void k_bvh_moments(const float4 *__restrict__ leaf_tris, int n, const rtb_bvhnode *__restrict__ nodes,
                              const int *__restrict__ parent_inner, const int *__restrict__ parent_leaf,
                              unsigned int *__restrict__ arrivals, float *__restrict__ moments)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    float t[12], N[3], c[3], r;
    for (int j = 0; j < 3; j++)
    {
        const float4 q = leaf_tris[3ull * p + j];
        t[4 * j] = q.x; t[4 * j + 1] = q.y; t[4 * j + 2] = q.z; t[4 * j + 3] = q.w;
    }
    rtb_winding::triMoment(t, N, c, r);
    auto store = [&](float *m) { m[0] = N[0]; m[1] = N[1]; m[2] = N[2]; m[3] = c[0]; m[4] = c[1]; m[5] = c[2]; m[6] = r; };
    if (n == 1)
    { // a single leaf: both slots of the root hold it
        store(moments);
        store(moments + 7);
        return;
    }
    int slot = parent_leaf[p];
    while (true)
    {
        const int node = slot >> 1, side = slot & 1;
        float *m = moments + 16ull * node;
        store(m + 7 * side);
        __threadfence();
        if (atomicAdd(arrivals + node, 1u) == 0u) return; // the sibling is still on its way: it continues
        __threadfence();
        float s[14];
        for (int j = 0; j < 14; j++) s[j] = __ldcg(m + j);
        const float *N0 = s, *c0 = s + 3, *N1 = s + 7, *c1 = s + 10;
        const float a0 = rtb_winding::norm3(N0), a1 = rtb_winding::norm3(N1), a = a0 + a1;
        for (int i = 0; i < 3; i++) N[i] = N0[i] + N1[i];
        if (a > 0.0f)
            for (int i = 0; i < 3; i++) c[i] = (c0[i] * a0 + c1[i] * a1) / a;
        else
        { // no area below: the centre of the node's box
            const rtb_bvhnode &b = nodes[node];
            for (int i = 0; i < 3; i++)
            {
                const float lo = b.lo[0][i] < b.lo[1][i] ? b.lo[0][i] : b.lo[1][i];
                const float hi = b.hi[0][i] > b.hi[1][i] ? b.hi[0][i] : b.hi[1][i];
                c[i] = (lo + hi) * 0.5f;
            }
        }
        const float d0[3] = {c[0] - c0[0], c[1] - c0[1], c[2] - c0[2]}, d1[3] = {c[0] - c1[0], c[1] - c1[1], c[2] - c1[2]};
        const float r0 = rtb_winding::norm3(d0) + s[6], r1 = rtb_winding::norm3(d1) + s[13];
        r = (r0 > r1 ? r0 : r1) * 1.00000095367431641f; // (1 + 2^-20): outward over the roundings
        if (node == 0) return;
        slot = parent_inner[node];
    }
}

} // namespace rtb
