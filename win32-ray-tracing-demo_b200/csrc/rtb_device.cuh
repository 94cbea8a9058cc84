// rtb_device.cuh -- device-side scene image and intersection routines (sm_100a).
//
// Arithmetic contract: every decision-making expression is IEEE float32 evaluated in the
// reference's operation order.  This translation unit is compiled with -fmad=false (no FMA
// contraction; the x86-64 reference build has none), default -prec-div/-prec-sqrt (correctly
// rounded / and sqrt) and -ftz=false.  Comparisons the reference performs in double against
// double literals are folded into the equivalent float thresholds:
//     fabs(x) <  1e-10 (double)  <=>  fabsf(x) <  1e-10f   (float(1e-10) is the least float >= 1e-10)
//     fabs(x) >  1e-10 (double)  <=>  fabsf(x) >= 1e-10f
//     fabs(x) >  0.1   (double)  <=>  fabsf(x) >= 0.1f     (float(0.1) is the least float >= 0.1)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>
#include "../../include/rtb.h"
#include "rtb_pretest.h"
#include "rtb_bvh.h"

#define RTB_MAX_INLINE_PRIMS 16
#define RTB_MAX_INLINE_MATS 16
#define RTB_KD_STACK 50 // reference Tunnel.cpp:1176

namespace rtb {

// ---------------------------------------------------------------------------------------------
// float3 algebra in the reference's operation order (Vector.cpp:48-86)
// ---------------------------------------------------------------------------------------------
struct V3 { float x, y, z; };
__device__ __forceinline__ V3 v3(float x, float y, float z) { V3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ V3 operator+(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ V3 operator-(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ V3 operator*(V3 a, float s) { return v3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ V3 mul(V3 a, V3 b) { return v3(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ V3 cross(V3 a, V3 b) { return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
__device__ __forceinline__ V3 normalize(V3 a) { return a * (1 / sqrtf(a.x * a.x + a.y * a.y + a.z * a.z)); }
__device__ __forceinline__ float comp(const V3 &a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }
// component by a RUN-TIME axis (the k-d walks): two selects instead of the compare-and-branch ladders the ternaries
// above turn into when the lanes of a warp sit on nodes with different split axes (11 instructions and a
// divergent region per pick in the SASS of the walk; 25 M inner nodes per 4K frame)
__device__ __forceinline__ float compSel(const V3 &a, int axis)
{
    float r;
    asm("{\n\t.reg .pred p;\n\tsetp.eq.s32 p, %4, 0;\n\tselp.f32 %0, %1, %2, p;\n\tsetp.eq.s32 p, %4, 2;\n\tselp.f32 %0, %3, %0, p;\n\t}"
        : "=f"(r) : "f"(a.x), "f"(a.y), "f"(a.z), "r"(axis));
    return r;
}
// v with component `axis` replaced by s (axis 3: v unchanged)
__device__ __forceinline__ V3 withComp(V3 v, int axis, float s)
{
    V3 r;
    asm("{\n\t.reg .pred p;\n\tsetp.eq.s32 p, %7, 0;\n\tselp.f32 %0, %6, %3, p;\n\tsetp.eq.s32 p, %7, 1;\n\tselp.f32 %1, %6, %4, p;\n\t"
        "setp.eq.s32 p, %7, 2;\n\tselp.f32 %2, %6, %5, p;\n\t}"
        : "=f"(r.x), "=f"(r.y), "=f"(r.z) : "f"(v.x), "f"(v.y), "f"(v.z), "f"(s), "r"(axis));
    return r;
}
__device__ __forceinline__ V3 ld3(const float *p) { return v3(p[0], p[1], p[2]); }

struct Ray { V3 o, d; };
__device__ __forceinline__ V3 at(const Ray &r, float t) { return r.o + r.d * t; } // Ray.h:24-27

// x86 cvttss2si semantics of the reference's (int) casts: out-of-range / NaN -> INT_MIN
__device__ __forceinline__ int f2i(float f)
{
    return (f >= -2147483648.0f && f < 2147483648.0f) ? (int)f : (int)0x80000000;
}

// ---------------------------------------------------------------------------------------------
// Device scene image.  Passed to kernels by value as a __grid_constant__ parameter: the handful
// of analytic primitives and materials live in the constant bank (warp-uniform reads), the
// triangle / accelerator streams are pointers into HBM (L2-resident after first touch).
// ---------------------------------------------------------------------------------------------
struct DScene
{
    int n_prims, n_materials, n_top, accel;
    rtb_prim prims[RTB_MAX_INLINE_PRIMS];
    rtb_material mats[RTB_MAX_INLINE_MATS];
    // triangles: 3 x float4 per triangle = {a.xyz, e1.x} {e1.yz, e2.xy} {e2.z, n.xyz},
    // e1 = a - b, e2 = a - c precomputed with the same float subtraction Triangle.cpp:73-79 does
    const float4 *loose;
    const float4 *tri;
    // the same triangles for the conservative rejection test (rtb_pretest.h): 3 x float4 = {a.xyz, A1 eps}
    // {e1.xyz, E eps} {e2.xyz, 0}, indexed by triangle; source of the pair stream below (k_pack_pairs).  The list
    // scans read the pair stream and touch `tri` only for candidates
    const float4 *tri_pre;
    // PAIR stream of the active accelerator's reference array (kd_tris or g_tris): for positions 2p and 2p + 1 six
    // float4 with the two triangles' rejection-test records interleaved component by component (rtb_pretest.h:
    // PreTri2, k_pack_pairs) -- what the packed FP32 scan reads, without index indirection.  null: linear / convex
    const float4 *pre2;
    const int *tri_material;
    int n_tris;
    // grid
    V3 g_origin, g_cell, g_far; // g_far = origin + cell * dims (Tunnel.cpp:822-825)
    V3 g_extent;                // cell * dims
    int nx, ny, nz;
    const uint2 *g_words;
    const uint32_t *g_start;
    const uint32_t *g_tris;
    // k-d
    V3 kd_min, kd_size; // Grid(near, far): pos = near, size = far - near (Grid.cpp:13-17)
    const uint2 *kd_nodes;
    const uint32_t *kd_tris;
    // convex accelerator (include/rtb.h: cx_*)
    int cx_n_path, cx_n_edges, cx_table, cx_round_bins;
    float cx_width, cx_height;
    const float *cx_frames;
    const float *cx_edges;
    const uint8_t *cx_status;
    const short *cx_range;
    const uint16_t *cx_order;
    // RTB_PRIM_MESH (rtb_build_bvh.cuh): every mesh record has its own slice of the three arrays, starting at
    // mesh_base[record index] (the mesh triangles of the records before it): its inner nodes at mesh_nodes[base ..]
    // (4 float4 each, the rtb_bvhnode layout), its triangles in leaf order at mesh_tris[base ..] (the exact stream's
    // format) and their local indices at mesh_order[base ..]
    const float4 *mesh_nodes;
    const float4 *mesh_tris;
    const uint32_t *mesh_order;
    int mesh_base[RTB_MAX_INLINE_PRIMS];
};

// Ray::context (reference Ray.h:11-16, RayContext.h:5-13): written by the convex accelerator, copied to the
// reflected ray by trace() (MainWindow.cpp:105, PerformanceTest/main.cpp:57)
struct RayCtx { int inTunnel, segment; };

struct Counters { unsigned long long rays, tris, steps, tiles; }; // tiles: finished tiles of the frame in flight (progress reporting)

// Probes: compile-time observation policy.  NoProbe costs nothing.
struct NoProbe
{
    __device__ __forceinline__ void step(int) {}
    __device__ __forceinline__ void tri() {}
};
struct CountProbe
{
    unsigned int tris = 0, steps = 0;
    __device__ __forceinline__ void step(int) { steps++; }
    __device__ __forceinline__ void tri() { tris++; }
};
struct SeqProbe
{ // records the traversal sequence of one primary ray
    int len = 0;
    unsigned long long hash = 0xcbf29ce484222325ull;
    int *buf = nullptr;
    int cap = 0;
    __device__ __forceinline__ void step(int id)
    {
        hash = (hash ^ (unsigned int)id) * 0x100000001b3ull;
        if (len < cap) buf[len] = id;
        len++;
    }
    __device__ __forceinline__ void tri() {}
};

// ---------------------------------------------------------------------------------------------
// Triangle -- reference Triangle.cpp:25-121 (Cramer's rule, four 3x3 determinants)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float det3(float a11, float a12, float a13, float a21, float a22, float a23,
                                      float a31, float a32, float a33)
{
    return a11 * a22 * a33 + a12 * a23 * a31 + a13 * a21 * a32 - a13 * a22 * a31 - a11 * a23 * a32 - a12 * a21 * a33;
}

struct TriData { float4 q0, q1, q2; };
__device__ __forceinline__ TriData loadTri(const float4 *base, unsigned int idx)
{
    const float4 *p = base + 3ull * idx;
    TriData t;
    t.q0 = __ldg(p);
    t.q1 = __ldg(p + 1);
    t.q2 = __ldg(p + 2);
    return t;
}
__device__ __forceinline__ V3 triNormal(const TriData &t) { return v3(t.q2.y, t.q2.z, t.q2.w); }
__device__ __forceinline__ rtb_pre::PreTri2 loadPreTri2(const float4 *base, unsigned int pair)
{
    const float4 *p = base + 6ull * pair;
    const float4 q0 = __ldg(p), q1 = __ldg(p + 1), q2 = __ldg(p + 2), q3 = __ldg(p + 3), q4 = __ldg(p + 4), q5 = __ldg(p + 5);
    rtb_pre::PreTri2 t;
    t.ax = make_float2(q0.x, q0.y); t.ay = make_float2(q0.z, q0.w); t.az = make_float2(q1.x, q1.y); t.a1e = make_float2(q1.z, q1.w);
    t.e1x = make_float2(q2.x, q2.y); t.e1y = make_float2(q2.z, q2.w); t.e1z = make_float2(q3.x, q3.y); t.ee = make_float2(q3.z, q3.w);
    t.e2x = make_float2(q4.x, q4.y); t.e2y = make_float2(q4.z, q4.w); t.e2z = make_float2(q5.x, q5.y);
    return t;
}

// ILP = false: the reference's statement order (exit after each quotient) -- fewest instructions, best
//               when the SM is issue-bound (the bulk of a frame);
// ILP = true : everything evaluated before one combined predicate -- best for latency-bound warps.
// Both produce the same values and the same accept / reject decisions.
template <bool ILP>
__device__ __forceinline__ bool triIntersectT(const TriData &T, const Ray &ray, float &tOut)
{
    const float m11 = T.q0.w, m21 = T.q1.x, m31 = T.q1.y; // a - b
    const float m12 = T.q1.z, m22 = T.q1.w, m32 = T.q2.x; // a - c
    const float m13 = ray.d.x, m23 = ray.d.y, m33 = ray.d.z;
    const float b1 = T.q0.x - ray.o.x, b2 = T.q0.y - ray.o.y, b3 = T.q0.z - ray.o.z;
    if (!ILP)
    {
    // the reference's statement order: four determinants with an exit after each quotient
    const float detM = det3(m11, m12, m13, m21, m22, m23, m31, m32, m33);
    if (fabsf(detM) < 1e-10f) return false;
    const float t = det3(m11, m12, b1, m21, m22, b2, m31, m32, b3) / detM;
    if (t < 0.0005f) return false;
    const float beta = det3(b1, m12, m13, b2, m22, m23, b3, m32, m33) / detM;
    if (beta < -0.0001f || beta > 1.0001f) return false;
    const float gamma = det3(m11, b1, m13, m21, b2, m23, m31, b3, m33) / detM;
    if (gamma < -0.0001f || gamma > 1.0001f || 1 - beta - gamma < -0.0001f || 1 - beta - gamma > 1.0001f) return false;
    tOut = t;
    return true;
    }
    // Same values, same accept / reject decisions, but all four determinants and the three quotients
    // are evaluated before any branch: the 48 multiplies and 20 adds are independent chains (ILP hides
    // the 4-cycle ALU latency that dominates a lone warp's stall cycles, profiles/r01_ncu_whitted_chain.md),
    // the reciprocal seed of det_m is shared by the three IEEE divisions, and the early exits become
    // one predicate.  The rejects are side-effect free, so evaluating past them cannot change a result;
    // quotients by a near-zero det_m are inf/NaN and discarded by the det test.
    const float detM = det3(m11, m12, m13, m21, m22, m23, m31, m32, m33);
    const float detT = det3(m11, m12, b1, m21, m22, b2, m31, m32, b3);
    const float detB = det3(b1, m12, m13, b2, m22, m23, b3, m32, m33);
    const float detG = det3(m11, b1, m13, m21, b2, m23, m31, b3, m33);
    const float t = detT / detM, beta = detB / detM, gamma = detG / detM;
    const float alpha = 1 - beta - gamma;
    const bool reject = (fabsf(detM) < 1e-10f) | (t < 0.0005f) | (beta < -0.0001f) | (beta > 1.0001f) |
                        (gamma < -0.0001f) | (gamma > 1.0001f) | (alpha < -0.0001f) | (alpha > 1.0001f);
    tOut = t;
    return !reject;
}
__device__ __forceinline__ bool triIntersect(const TriData &T, const Ray &ray, float &tOut) { return triIntersectT<false>(T, ray, tOut); }

// nearest hit of a list of triangle references; first in list wins ties (strict <)
// WIDE = false: one lane walks the list (the lanes of a warp hold different rays).
// WIDE = true : the whole warp holds ONE ray (rtb_chain_wide.cuh) and tests 32 triangles of the list at a
//               time, one per lane; the nearest accepted hit is found with a warp min-reduction, ties go to
//               the earliest list position as in the sequential scan.  Every lane returns the same result.
template <bool WINDOW, bool WIDE, class Probe>
__device__ __forceinline__ bool nearestInList(const DScene &S, const uint32_t *refs, uint32_t first, uint32_t last,
                                              const Ray &ray, float lo, float hi, int &triOut, float &tOut,
                                              V3 &nOut, Probe &pr)
{
    float minDistance = FLT_MAX;
    bool found = false;
    if constexpr (WIDE)
    {
        const uint32_t lane = threadIdx.x & 31u;
        for (uint32_t base = first; base < last; base += 32)
        {
            const uint32_t i = base + lane;
            float t = FLT_MAX;
            uint32_t idx = 0;
            bool ok = false;
            if (i < last)
            {
                idx = __ldg(refs + i);
                const TriData T = loadTri(S.tri, idx);
                pr.tri();
                ok = triIntersectT<true>(T, ray, t);
                if (WINDOW) ok = ok && (t >= lo && t <= hi);
                ok = ok && t < FLT_MAX; // an accepted t is >= 0.0005; inf / NaN never become a hit in the reference either
            }
            // accepted distances are positive floats: their bit patterns order like the values
            const uint32_t key = ok ? __float_as_uint(t) : 0xffffffffu;
            const uint32_t best = __reduce_min_sync(0xffffffffu, key);
            if (best != 0xffffffffu && __uint_as_float(best) < minDistance)
            { // strict <: an equal distance in a later group of 32 does not replace the earlier one
                const uint32_t who = __ffs(__ballot_sync(0xffffffffu, key == best)) - 1; // earliest list position
                minDistance = __uint_as_float(best);
                triOut = (int)__shfl_sync(0xffffffffu, idx, who);
                found = true;
            }
        }
        if (found)
        {
            const float4 q2 = __ldg(S.tri + 3ull * (unsigned int)triOut + 2);
            nOut = v3(q2.y, q2.z, q2.w);
        }
        tOut = minDistance;
        return found;
    }
    else
    {
        // Per-lane scan.  Every list entry first meets the conservative rejection test (rtb_pretest.h: the four
        // determinants by two cross products with FMA, no division, plus an error bound; no data-dependent branch),
        // two entries per iteration on the packed FP32 pipe, read from the pair stream (no index indirection): list
        // positions 2p and 2p + 1 form pair p, a list that starts or ends on an odd position masks the foreign half.
        // The test never accepts: an entry it cannot reject is a CANDIDATE and takes the reference's exact test, so
        // results are bit-identical.  Candidates are essentially the ray's real hits (1.06-1.6 per ray,
        // profiles/r01_pretest_stats.md), so their exact test is DEFERRED to the end of the list: inside the loop it
        // would be executed -- by warp union -- in most iterations for the one lane that needs it.  Should a second
        // candidate turn up while one is pending (0.1-0.3 % of the lists) the fast loop stops and the rest of the
        // list is scanned exactly, in order.
        const float dmx = rtb_pre::dirMax(ray.d.x, ray.d.y, ray.d.z);
        const float Lp = rtb_pre::lowBound(WINDOW ? lo : -FLT_MAX);
        const float Hp = rtb_pre::highBound(WINDOW ? hi : FLT_MAX, FLT_MAX);
        uint32_t pend = 0xffffffffu;
        uint32_t counted = last; // list positions below `counted` have gone through pr.tri()
        bool multi = false;      // the fast loop stopped at a second candidate
        const uint32_t pEnd = (last + 1u) >> 1;
        for (uint32_t p = first >> 1; p < pEnd; p++)
        {
            const rtb_pre::PreTri2 P = loadPreTri2(S.pre2, p);
            const uint32_t j0 = 2u * p, j1 = j0 + 1u;
            const bool in0 = j0 >= first, in1 = j1 < last; // j0 < last and j1 >= first always hold
            if (in0) pr.tri();
            if (in1) pr.tri();
            bool r0, r1;
            rtb_pre::sureReject2<WINDOW>(P, ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z, dmx, Lp, Hp, r0, r1);
            const bool c0 = in0 && !r0, c1 = in1 && !r1;
            if (!(c0 || c1)) continue;
            if (pend != 0xffffffffu || (c0 && c1))
            { // a second candidate: exact scan from the first one to the end of the list
                if (pend == 0xffffffffu) pend = j0;
                counted = in1 ? j1 + 1u : j1;
                multi = true;
                break;
            }
            pend = c0 ? j0 : j1;
        }
        if (pend != 0xffffffffu)
        {
            // [pend, pend + 1) when the fast loop ran to the end, else [pend, last): entries the fast loop proved
            // rejects are tested again on the way, which changes nothing
            const uint32_t jend = multi ? last : pend + 1;
            for (uint32_t j = pend; j < jend; j++)
            {
                const uint32_t idx = __ldg(refs + j);
                const TriData T = loadTri(S.tri, idx);
                if (j >= counted) pr.tri();
                float t;
                if (!triIntersect(T, ray, t)) continue;
                if (WINDOW && !(t >= lo && t <= hi)) continue;
                if (t < minDistance)
                {
                    minDistance = t;
                    triOut = (int)idx;
                    nOut = triNormal(T);
                    found = true;
                }
            }
        }
        tOut = minDistance;
        return found;
    }
}

// ---------------------------------------------------------------------------------------------
// Box entry / exit -- reference Grid.cpp:30-116
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void updateEntryExit(float &entry, float &exit, float v)
{
    if (entry == FLT_MAX && exit == FLT_MAX) entry = v;
    else if (exit == FLT_MAX)
    {
        if (v > entry) exit = v;
        else { exit = entry; entry = v; }
    }
    else
    {
        if (v < entry) { exit = entry; entry = v; }
        else if (v < exit) exit = v;
    }
}

__device__ __forceinline__ void boxFace(float planePos, float o, float d, const Ray &ray, int a1, int a2,
                                        const V3 &nearP, const V3 &farP, float &entry, float &exit)
{
    const float distance = (planePos - o) / d;
    const V3 p = at(ray, distance);
    const float u = comp(p, a1), v = comp(p, a2);
    if (u >= comp(nearP, a1) && u <= comp(farP, a1) && v >= comp(nearP, a2) && v <= comp(farP, a2))
        updateEntryExit(entry, exit, distance);
}

__device__ __forceinline__ bool boxIntersect(V3 nearP, V3 size, const Ray &ray, float &entry, float &exit)
{
    const V3 farP = nearP + size;
    entry = FLT_MAX;
    exit = FLT_MAX;
    if (fabsf(ray.d.x) >= 1e-10f)
    {
        boxFace(nearP.x, ray.o.x, ray.d.x, ray, 1, 2, nearP, farP, entry, exit);
        boxFace(farP.x, ray.o.x, ray.d.x, ray, 1, 2, nearP, farP, entry, exit);
    }
    if (fabsf(ray.d.y) >= 1e-10f)
    {
        boxFace(nearP.y, ray.o.y, ray.d.y, ray, 2, 0, nearP, farP, entry, exit);
        boxFace(farP.y, ray.o.y, ray.d.y, ray, 2, 0, nearP, farP, entry, exit);
    }
    if (fabsf(ray.d.z) >= 1e-10f)
    {
        boxFace(nearP.z, ray.o.z, ray.d.z, ray, 0, 1, nearP, farP, entry, exit);
        boxFace(farP.z, ray.o.z, ray.d.z, ray, 0, 1, nearP, farP, entry, exit);
    }
    return entry != FLT_MAX;
}

// ---------------------------------------------------------------------------------------------
// Grid 3D-DDA -- reference Tunnel.cpp:806-970
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void indexInGrid(const DScene &S, V3 p, int &i, int &j, int &k)
{
    i = f2i((p.x - S.g_origin.x) / S.g_cell.x);
    j = f2i((p.y - S.g_origin.y) / S.g_cell.y);
    k = f2i((p.z - S.g_origin.z) / S.g_cell.z);
    if (i < 0) i = 0;
    if (j < 0) j = 0;
    if (k < 0) k = 0;
    if (i > S.nx - 1) i = S.nx - 1;
    if (j > S.ny - 1) j = S.ny - 1;
    if (k > S.nz - 1) k = S.nz - 1;
}

template <bool WIDE, class Probe>
__device__ bool gridIntersect(const DScene &S, const Ray &ray, int &triOut, float &tOut, V3 &nOut, Probe &pr)
{
    int ci, cj, ck;
    float cd;
    V3 cp;
    if (ray.o.x < S.g_origin.x || ray.o.x > S.g_far.x || ray.o.y < S.g_origin.y || ray.o.y > S.g_far.y ||
        ray.o.z < S.g_origin.z || ray.o.z > S.g_far.z)
    {
        float entry, exit;
        if (!boxIntersect(S.g_origin, S.g_extent, ray, entry, exit)) return false;
        cd = entry;
        cp = at(ray, entry);
        indexInGrid(S, cp, ci, cj, ck);
    }
    else
    {
        cp = ray.o;
        cd = 0;
        indexInGrid(S, ray.o, ci, cj, ck);
    }
    const bool px = ray.d.x > 0, py = ray.d.y > 0, pz = ray.d.z > 0;
    while (true)
    {
        const int cell = (ci * S.ny + cj) * S.nz + ck;
        pr.step(cell);
        const uint2 w = __ldg(S.g_words + ((unsigned int)cell >> 5));
        const unsigned int bit = 1u << (cell & 31);
        if (w.x & bit)
        {
            const unsigned int r = w.y + __popc(w.x & (bit - 1));
            const uint32_t first = __ldg(S.g_start + r), last = __ldg(S.g_start + r + 1);
            if (nearestInList<false, WIDE>(S, S.g_tris, first, last, ray, 0.f, 0.f, triOut, tOut, nOut, pr)) return true;
        }
        // distance to the exit plane of the current cell on each axis; cell corners are recomputed
        // from the integer indices every step (Tunnel.cpp:885-938); IEEE inf/NaN semantics kept
        float dx, dy, dz;
        if (px) dx = ((S.g_origin.x + (ci + 1) * S.g_cell.x) - cp.x) / ray.d.x;
        else dx = (cp.x - (S.g_origin.x + ci * S.g_cell.x)) / -ray.d.x;
        if (py) dy = ((S.g_origin.y + (cj + 1) * S.g_cell.y) - cp.y) / ray.d.y;
        else dy = (cp.y - (S.g_origin.y + cj * S.g_cell.y)) / -ray.d.y;
        if (pz) dz = ((S.g_origin.z + (ck + 1) * S.g_cell.z) - cp.z) / ray.d.z;
        else dz = (cp.z - (S.g_origin.z + ck * S.g_cell.z)) / -ray.d.z;
        if (dx < dy && dx < dz) { ci += px ? 1 : -1; cd += dx; }
        else if (dy < dz) { cj += py ? 1 : -1; cd += dy; }
        else { ck += pz ? 1 : -1; cd += dz; }
        cp = at(ray, cd);
        if (ci < 0 || ci > S.nx - 1 || cj < 0 || cj > S.ny - 1 || ck < 0 || ck > S.nz - 1) break;
    }
    return false;
}

// ---------------------------------------------------------------------------------------------
// k-d tree -- reference Tunnel.cpp:1163-1297 (Havran TA_rec_B).
// The reference keeps {node, t, pb, prev} per stack element.  pb is a pure function of
// (t, axis, split): pb[axis] = split, pb[other] = o + t*d (lines 1260-1262), so an element is
// stored as 16 bytes {node, t, split, axis | prev<<2} and pb is re-derived bit-exactly when the
// element becomes the exit point again.  The current entry/exit elements live in registers.
// axis code 3 = "all three components are o + t*d" (the initial exit point, line 1196).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ V3 kdPoint(const Ray &ray, float t, float split, int axis)
{
    return withComp(v3(ray.o.x + t * ray.d.x, ray.o.y + t * ray.d.y, ray.o.z + t * ray.d.z), axis, split);
}

template <bool WIDE, class Probe>
__device__ bool kdIntersect(const DScene &S, const Ray &ray, int &triOut, float &tOut, V3 &nOut, Probe &pr)
{
    float a, b;
    if (!boxIntersect(S.kd_min, S.kd_size, ray, a, b)) return false;
    int4 stack[RTB_KD_STACK];
    // entry point (element 0)
    float enT = a;
    V3 enP = (a >= 0) ? (ray.o + ray.d * a) : ray.o;
    int enPt = 0;
    // exit point (element 1), node -1 = termination flag
    int exPt = 1;
    float exT = b;
    V3 exP = ray.o + ray.d * b;
    int exNode = -1, exPrev = 0;
    stack[1] = make_int4(-1, __float_as_int(b), 0, 3);
    int cur = 0;
    while (cur != -1)
    {
        uint2 nd = __ldg(S.kd_nodes + cur);
        while ((nd.y & 3u) != 3u)
        {
            pr.step(cur);
            const float splitVal = __uint_as_float(nd.x);
            const int axis = (int)(nd.y & 3u);
            const int right = (int)(nd.y >> 2), left = cur + 1;
            const float en = compSel(enP, axis), ex = compSel(exP, axis);
            int farChild;
            if (en <= splitVal)
            {
                if (ex <= splitVal) { cur = left; nd = __ldg(S.kd_nodes + cur); continue; }
                if (ex == splitVal) { cur = right; nd = __ldg(S.kd_nodes + cur); continue; } // unreachable, kept for fidelity (line 1223)
                farChild = right; cur = left;
            }
            else
            {
                if (splitVal < ex) { cur = right; nd = __ldg(S.kd_nodes + cur); continue; }
                farChild = left; cur = right;
            }
            const float t = (splitVal - compSel(ray.o, axis)) / compSel(ray.d, axis);
            const int tmp = exPt++;
            if (exPt == enPt) exPt += 1;
            exPrev = tmp; exT = t; exNode = farChild;
            exP = kdPoint(ray, t, splitVal, axis);
            stack[exPt] = make_int4(farChild, __float_as_int(t), __float_as_int(splitVal), axis | (tmp << 2));
            nd = __ldg(S.kd_nodes + cur);
        }
        pr.step(cur);
        const uint32_t first = nd.x, count = nd.y >> 2;
        if (count && nearestInList<true, WIDE>(S, S.kd_tris, first, first + count, ray, enT - 0.001f, exT + 0.001f,
                                         triOut, tOut, nOut, pr))
            return true;
        // pop: the signed distance intervals are adjacent
        enPt = exPt; enT = exT; enP = exP;
        cur = exNode;
        if (cur == -1) break;
        exPt = exPrev;
        const int4 e = stack[exPt];
        exNode = e.x; exT = __int_as_float(e.y); exPrev = e.w >> 2;
        exP = kdPoint(ray, exT, __int_as_float(e.z), e.w & 3);
    }
    return false;
}

template <class Probe>
__device__ bool linearIntersect(const DScene &S, const Ray &ray, int &triOut, float &tOut, V3 &nOut, Probe &pr)
{ // reference Tunnel.cpp:786-804
    float minDistance = FLT_MAX;
    bool found = false;
    for (int i = 0; i < S.n_tris; i++)
    {
        const TriData T = loadTri(S.tri, i);
        pr.tri();
        float t;
        if (triIntersect(T, ray, t) && t < minDistance) { minDistance = t; triOut = i; nOut = triNormal(T); found = true; }
    }
    tOut = minDistance;
    return found;
}

// ---------------------------------------------------------------------------------------------
// Convex accelerator -- reference PerformanceTest/ConvexAcc.cpp:7-84, 273-415 (Tunnel.cpp:972-1161).
// A ray inside the tunnel walks from cross-section polygon to polygon (point-in-convex-polygon through the
// lookup table) until it leaves through the wall of a segment, then tries that segment's triangles in
// list order (ConvexSimple) or in the order of the (height, direction) table (Convex) and returns the FIRST
// accepted one.  All tables come from the host (rtb_scene_upload); what runs here is float arithmetic in the
// reference's order plus one atan2f per wall exit (CUDA's differs from glibc's in the last ulps: it can
// select the neighbouring direction bin only when the angle sits on a bin boundary to within those ulps).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ bool convexAtOrigin(const DScene &S, V3 o, V3 d, float &distance)
{
    if (o.z * d.z >= 0) return false;
    distance = (0 - o.z) / d.z;
    const V3 p = o + d * distance;
    const int table = S.cx_table; // 100 (PerformanceTest) or 400 (RayTracingOpt)
    const float cellWidth = S.cx_width / (table - 1.0f), cellHeight = S.cx_height / (table - 1.0f);
    int i = f2i((p.x + S.cx_width / 2) / cellWidth + 0.5f), j = f2i(p.y / cellHeight + 0.5f);
    i = max(i, 0); j = max(j, 0);
    i = min(i, table - 1); j = min(j, table - 1);
    const int cell = i * table + j;
    const unsigned int st = __ldg(S.cx_status + cell);
    if (st == 0) return true;
    if (st == 2) return false;
    const int begin = __ldg(S.cx_range + 2 * cell), end = __ldg(S.cx_range + 2 * cell + 1);
    for (int e = begin; e <= end; e++)
        if (__ldg(S.cx_edges + 3 * e) * p.x + __ldg(S.cx_edges + 3 * e + 1) * p.y + __ldg(S.cx_edges + 3 * e + 2) < 0.0001f) return false;
    return true;
}

__device__ __forceinline__ bool convexPolygon(const DScene &S, const Ray &ray, int index, V3 &origin, V3 &dir, float &distance)
{
    const float *f = S.cx_frames + 8 * index;
    const float c = __ldg(f + 6), s = __ldg(f + 7);
    const V3 q = v3(ray.o.x + (0 - __ldg(f)), ray.o.y + (0 - __ldg(f + 1)), ray.o.z + (0 - __ldg(f + 2)));
    V3 newOrigin = v3(c * q.x + 0 * q.y + s * q.z, 0 * q.x + 1 * q.y + 0 * q.z, -s * q.x + 0 * q.y + c * q.z);
    V3 newDir = v3(c * ray.d.x + 0 * ray.d.y + s * ray.d.z, 0 * ray.d.x + 1 * ray.d.y + 0 * ray.d.z, -s * ray.d.x + 0 * ray.d.y + c * ray.d.z);
    const bool hit = convexAtOrigin(S, newOrigin, newDir, distance);
    if (!hit)
    {
        newOrigin.z = 0;
        newDir.z = 0;
        origin = newOrigin;
        dir = normalize(newDir);
    }
    return hit;
}

template <class Probe>
__device__ bool convexIntersect(const DScene &S, const Ray &ray, RayCtx &ctx, int &triOut, float &tOut, V3 &nOut, Probe &pr)
{
    Ray adv = ray;
    float distance = 0;
    const int N = S.cx_n_path - 1;
    const int perSegment = 2 * S.cx_n_edges;
    auto ringNormal = [&](int i) { return v3(__ldg(S.cx_frames + 8 * i + 3), __ldg(S.cx_frames + 8 * i + 4), __ldg(S.cx_frames + 8 * i + 5)); };
    if (!ctx.inTunnel)
    {
        V3 no, nd;
        if (convexPolygon(S, ray, 0, no, nd, distance) && dot(ray.d, ringNormal(0)) > 0)
        { // through the entrance
            ctx.inTunnel = 1; ctx.segment = 0;
            adv.o = at(ray, distance);
        }
        else if (convexPolygon(S, ray, N, no, nd, distance) && dot(ray.d, ringNormal(N)) < 0)
        { // through the exit
            ctx.inTunnel = 1; ctx.segment = N - 1;
            adv.o = at(ray, distance);
        }
        else return linearIntersect(S, ray, triOut, tOut, nOut, pr); // starts outside and never enters
    }
    const int begin = ctx.segment;
    if (!(dot(ray.d, ringNormal(begin)) > 0)) return false; // "Backward" is unimplemented in the reference (ConvexAcc.cpp:405-410)
    for (int i = begin + 1; i <= N; i++)
    {
        V3 no, nd;
        if (!convexPolygon(S, adv, i, no, nd, distance))
        { // the ray leaves through the wall of segment i - 1
            const int base = (i - 1) * perSegment;
            const uint16_t *row = nullptr;
            if (S.accel == RTB_ACCEL_CONVEX)
            {
                const float y = no.y - no.x * nd.y / nd.x;
                int index = f2i(99.0f * y / S.cx_height + 0.5f);
                index = max(0, index); index = min(99, index);
                const float PI_F = 3.14159265359f;
                float fAngle = atan2f(nd.y, nd.x);
                fAngle = (fAngle < 0) ? fAngle + PI_F * 2 : fAngle;
                int iAngle = S.cx_round_bins ? f2i(fAngle / PI_F * 180.0f + 0.5f) % 360 : f2i(fAngle / PI_F * 180.0f);
                iAngle = max(0, iAngle); iAngle = min(359, iAngle);
                row = S.cx_order + ((size_t)index * 360 + iAngle) * perSegment;
            }
            for (int j = 0; j < perSegment; j++)
            {
                const int idx = base + (row ? (int)__ldg(row + j) : j);
                const TriData T = loadTri(S.tri, idx);
                pr.tri();
                float t;
                if (triIntersect(T, ray, t))
                {
                    ctx.segment = i - 1;
                    triOut = idx; tOut = t; nOut = triNormal(T);
                    return true;
                }
            }
            if (S.accel == RTB_ACCEL_CONVEX) adv.o = at(adv, distance); // ConvexSimple does not advance here (lines 358-371)
        }
        else adv.o = at(adv, distance);
    }
    ctx.inTunnel = 0;
    return false;
}

// ---------------------------------------------------------------------------------------------
// Triangle mesh (RTB_PRIM_MESH): the hierarchy of rtb_build_bvh.cuh, nodes skipped by the test of rtb_bvh.h.  Nearest
// accepted (t, k) in lexicographic order; `bestT` comes in as the nearest hit of the earlier records and `bestK` as -1, so
// the mesh replaces it only with a strictly smaller t, as the run's `t < minDistance` does.  Visit order changes nothing.
// ANY = true (occlusion queries): the walk ends at the first accepted triangle with t < bestT; bestT / bestK / nOut are then
// that triangle's, not the nearest one's.
// ---------------------------------------------------------------------------------------------
template <bool ANY = false, class Probe>
__device__ bool meshIntersect(const DScene &S, unsigned int base, const Ray &ray, float &bestT, int &bestK, V3 &nOut, Probe &pr)
{
    const rtb_bvh::Ray R = rtb_bvh::makeRay(ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z);
    const float4 *nodes = S.mesh_nodes + 4ull * base;
    int stack[RTB_BVH_STACK];
    int sp = 0, node = 0;
    bool found = false;
    auto leaf = [&](int pos) {
        const TriData T = loadTri(S.mesh_tris, base + (unsigned int)pos);
        pr.tri();
        float t;
        if (!triIntersect(T, ray, t)) return;
        const int k = (int)__ldg(S.mesh_order + base + pos);
        if (t < bestT || (t == bestT && k < bestK)) { bestT = t; bestK = k; nOut = triNormal(T); found = true; }
    };
    while (true)
    {
        pr.step(node);
        const float4 *q = nodes + 4ull * (unsigned int)node;
        const float4 q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2), q3 = __ldg(q + 3);
        const float lo0[3] = {q0.x, q0.y, q0.z}, lo1[3] = {q0.w, q1.x, q1.y};
        const float hi0[3] = {q1.z, q1.w, q2.x}, hi1[3] = {q2.y, q2.z, q2.w};
        const int c0 = __float_as_int(q3.x), c1 = __float_as_int(q3.y);
        const bool h0 = rtb_bvh::nodeHit(R, lo0, hi0, bestT);
        const bool h1 = c1 != c0 && rtb_bvh::nodeHit(R, lo1, hi1, bestT); // a one-triangle mesh links its leaf twice
        if (h0 && c0 < 0) leaf(~c0);
        if (h1 && c1 < 0) leaf(~c1);
        if (ANY && found) break;
        const bool in0 = h0 && c0 >= 0, in1 = h1 && c1 >= 0;
        if (in0 && in1) { stack[sp++] = c1; node = c0; }
        else if (in0) node = c0;
        else if (in1) node = c1;
        else if (sp > 0) node = stack[--sp];
        else break;
    }
    return found;
}

// ---------------------------------------------------------------------------------------------
// GeometrySet::intersect -- reference GeometrySet.cpp:95-110 (+ Plane.cpp:9-34, Sphere.cpp:10-37)
// ---------------------------------------------------------------------------------------------
struct Hit { int id; int mat; int prim_type; float t; V3 pos, n; };

// `tunnel(tri, t, n)` supplies the result of the TUNNEL geometry (a traversal, or a result computed
// earlier by the resumable traversal of rtb_chain_sm.cuh); everything else is evaluated here in
// insertion order with the reference's strict `<`.
// MESH = false: scenes without RTB_PRIM_MESH records (the kernels every other scene runs are compiled without the mesh walk)
// `start`: the search starts there instead of at FLT_MAX, so every record's strict `<` rejects hits at t >= start (the
// bounded queries of rtb_query_rays; callers pass at most FLT_MAX).
// ANY = true: occlusion -- true as soon as one record has a hit with t < start (the minimum over the records is below start
// then, whatever the others hold); `best` is not filled.  The records are taken in order with the tunnel last, the TRIANGLES
// runs and the mesh walk stop at their first accepted triangle, the tunnel runs its closest walk (DESIGN 3d).
template <bool MESH = false, bool ANY = false, class Probe, class TunnelFn>
__device__ __forceinline__ bool sceneIntersectWith(const DScene &S, const Ray &ray, Hit &best, Probe &pr, TunnelFn tunnel,
                                                   float start = FLT_MAX)
{
    float minDistance = start;
    best.id = -1;
    bool tunnelLast = false;
    for (int i = 0; i < S.n_prims; i++)
    {
        const rtb_prim &P = S.prims[i];
        if (ANY && best.id >= 0) return true;
        if (P.type == RTB_PRIM_PLANE)
        {
            const V3 normal = v3(P.v[0], P.v[1], P.v[2]);
            const V3 op = v3(P.v[3], P.v[4], P.v[5]) - ray.o;
            const bool back = dot(normal, op) > 0;
            const V3 n = back ? normal : normal * -1;
            if (dot(n, ray.d) > 0)
            {
                const float distance = dot(op, n) / dot(ray.d, n);
                if (distance >= 0.0005f && distance < minDistance)
                {
                    minDistance = distance;
                    best.id = P.base_id; best.mat = P.material; best.n = normal; best.prim_type = RTB_PRIM_PLANE;
                }
            }
        }
        else if (P.type == RTB_PRIM_SPHERE)
        {
            const V3 center = v3(P.v[0], P.v[1], P.v[2]);
            const float radius = P.v[3];
            const V3 co = ray.o - center;
            const float b = dot(ray.d, co);
            float delta = b * b - (dot(co, co) - radius * radius);
            if (delta >= 0)
            {
                delta = sqrtf(delta);
                if (-b + delta >= 0.0005f)
                {
                    const float distance = (-b - delta >= 0.0005f) ? -b - delta : -b + delta;
                    if (distance < minDistance)
                    {
                        minDistance = distance;
                        best.id = P.base_id; best.mat = P.material; best.prim_type = RTB_PRIM_SPHERE;
                        best.n = normalize(at(ray, distance) - center);
                    }
                }
            }
        }
        else if (P.type == RTB_PRIM_TRIANGLES)
        {
            for (int k = 0; k < P.count; k++)
            {
                const TriData T = loadTri(S.loose, P.first + k);
                pr.tri();
                float t;
                if (triIntersect(T, ray, t) && t < minDistance)
                {
                    if (ANY) return true;
                    minDistance = t;
                    best.id = P.base_id + k; best.mat = P.material; best.n = triNormal(T); best.prim_type = RTB_PRIM_TRIANGLES;
                }
            }
        }
        else if (MESH && P.type == RTB_PRIM_MESH)
        {
            int k = -1;
            V3 n;
            if (meshIntersect<ANY>(S, (unsigned int)S.mesh_base[i], ray, minDistance, k, n, pr))
            {
                best.id = P.base_id + k; best.mat = P.material; best.n = n; best.prim_type = RTB_PRIM_MESH;
            }
        }
        else if (ANY) tunnelLast = true;
        else
        {
            int tri = -1;
            float t;
            V3 n;
            const bool ok = tunnel(tri, t, n);
            if (ok && t < minDistance)
            {
                minDistance = t;
                best.id = S.n_top + tri; best.mat = __ldg(S.tri_material + tri); best.n = n; best.prim_type = RTB_PRIM_TUNNEL;
            }
        }
    }
    if (ANY)
    {
        if (best.id >= 0) return true;
        if (!tunnelLast) return false;
        int tri = -1;
        float t;
        V3 n;
        return tunnel(tri, t, n) && t < minDistance;
    }
    if (best.id < 0) return false;
    best.t = minDistance;
    best.pos = at(ray, minDistance);
    return true;
}

template <bool MESH = false, bool ANY = false, class Probe>
__device__ bool sceneIntersect(const DScene &S, const Ray &ray, Hit &best, Probe &pr, RayCtx &ctx, float start = FLT_MAX)
{
    return sceneIntersectWith<MESH, ANY>(S, ray, best, pr, [&](int &tri, float &t, V3 &n) {
        if (S.accel == RTB_ACCEL_REGULAR_GRID || S.accel == RTB_ACCEL_FLAT_GRID) return gridIntersect<false>(S, ray, tri, t, n, pr);
        if (S.accel == RTB_ACCEL_KD_MEDIAN || S.accel == RTB_ACCEL_KD_SAH) return kdIntersect<false>(S, ray, tri, t, n, pr);
        if (S.accel == RTB_ACCEL_CONVEX || S.accel == RTB_ACCEL_CONVEX_SIMPLE) return convexIntersect(S, ray, ctx, tri, t, n, pr);
        return linearIntersect(S, ray, tri, t, n, pr);
    }, start);
}
// a ray generated by the camera or by a caller carries a fresh context
template <bool MESH = false, bool ANY = false, class Probe>
__device__ bool sceneIntersect(const DScene &S, const Ray &ray, Hit &best, Probe &pr, float start = FLT_MAX)
{
    RayCtx ctx;
    ctx.inTunnel = 0; ctx.segment = -1;
    return sceneIntersect<MESH, ANY>(S, ray, best, pr, ctx, start);
}

// ---------------------------------------------------------------------------------------------
// Camera -- reference Camera.cpp:20-26
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ Ray generateRay(const rtb_camera &c, float x, float y)
{
    const V3 right = ld3(c.right), up = ld3(c.up), front = ld3(c.front), eye = ld3(c.eye);
    const V3 r = right * ((x - c.xcenter) * c.fov_scale);
    const V3 u = up * ((y - 0.5f) * c.fov_scale);
    const V3 dir = normalize(front + r + u);
    Ray ray;
    ray.o = eye + dir * c.forward;
    ray.d = dir;
    return ray;
}

// ---------------------------------------------------------------------------------------------
// Materials -- reference *Material.cpp
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float checkerParity(const rtb_material &m, V3 pos)
{ // CheckerMaterial.cpp:13-21; d is a non-negative integer-valued float, so fmod(d, 2) is exact
    float d;
    if (m.dir == RTB_DIR_XOZ) d = fabsf(floorf(pos.x * m.scale) + floorf(pos.z * m.scale));
    else if (m.dir == RTB_DIR_YOZ) d = fabsf(floorf(pos.y * m.scale) + floorf(pos.z * m.scale));
    else d = fabsf(floorf(pos.x * m.scale) + floorf(pos.y * m.scale));
    return fmodf(d, 2.0f);
}

__device__ __forceinline__ V3 matLocal(const rtb_material &m, const Ray &ray, V3 pos, V3 normal)
{
    if (m.kind == RTB_MAT_SOLID) return ld3(m.a);
    if (m.kind == RTB_MAT_CHECKER) return checkerParity(m, pos) < 1 ? v3(0.15f, 0.15f, 0.15f) : v3(1, 1, 1);
    if (m.kind == RTB_MAT_RADIANCE_CHECKER) return v3(0.15f, 0.15f, 0.15f);
    // PhongMaterial.cpp:13-29: stored (unflipped) normal, white light from normalize(-1,1,1)
    const V3 lightDir = normalize(v3(-1, 1, 1));
    float NdotL = dot(normal, lightDir);
    NdotL = (NdotL < 0.0f) ? 0.0f : NdotL;
    const V3 H = normalize(lightDir - ray.d);
    float NdotH = dot(normal, H);
    NdotH = (NdotH < 0.0f) ? 0.0f : NdotH;
    const V3 diffuseTerm = ld3(m.a) * NdotL;
    const V3 specularTerm = ld3(m.b) * powf(NdotH, m.p);
    return mul(v3(1, 1, 1), diffuseTerm + specularTerm);
}

__device__ __forceinline__ V3 matEmission(const rtb_material &m, V3 pos)
{
    if (m.kind == RTB_MAT_SOLID) return ld3(m.b);
    if (m.kind == RTB_MAT_RADIANCE_CHECKER) return checkerParity(m, pos) < 1 ? v3(m.p, m.p, m.p) : v3(0, 0, 0);
    return v3(0, 0, 0);
}

// Refraction set-up shared by trace() and radiance() -- reference MainWindow.cpp:111-133 == 212-231
struct Fresnel { V3 refl, tdir; bool tir; float Re, Tr, P, RP, TP; };
__device__ __forceinline__ Fresnel refraction(const Ray &r, V3 n, V3 nl, float nt)
{
    Fresnel f;
    f.refl = r.d - n * 2 * dot(n, r.d);
    const bool into = dot(n, nl) > 0;
    const float nc = 1;
    const float nnt = into ? nc / nt : nt / nc;
    const float ddn = dot(r.d, nl);
    const float cos2t = 1 - nnt * nnt * (1 - ddn * ddn);
    f.tir = cos2t < 0;
    f.tdir = v3(0, 0, 0);
    f.Re = f.Tr = f.P = f.RP = f.TP = 0;
    if (f.tir) return f;
    f.tdir = normalize(r.d * nnt - n * ((into ? 1 : -1) * (ddn * nnt + sqrtf(cos2t))));
    const float a = nt - nc, b = nt + nc;
    const float R0 = a * a / (b * b);
    const float c = 1 - (into ? -ddn : dot(f.tdir, n));
    f.Re = R0 + (1 - R0) * c * c * c * c * c;
    f.Tr = 1 - f.Re;
    f.P = 0.25f + 0.5f * f.Re;
    f.RP = f.Re / f.P;
    f.TP = f.Tr / (1 - f.P);
    return f;
}

// ---------------------------------------------------------------------------------------------
// Counter-based RNG: Philox4x32-10, key = (pixel, sample), counter = (block, seed_lo, seed_hi, 0).
// Replaces the reference's per-row erand48 stream (erand48.h:53-81, MainWindow.cpp:273), which is
// inherently sequential; statistical parity only (oracle/rt_oracle.cpp mirrors this stream in its
// ORACLE_RNG_COUNTER mode so paths can also be compared one to one).
// ONE block per traced ray: block 0 of a sample carries the pixel jitter (slots 0, 1), block k belongs to the
// k-th ray of the sample, and the four values are addressed by slot -- 0 Russian roulette, 1 p_type, 2 / 3 the
// hemisphere pair, 2 the reflect-or-transmit test.  Every lane computes its block at the same point of the
// loop; with a sequential stream each lane refilled at its own time and the ten rounds ran up to four times
// per warp and vertex, from an inlined copy at every draw site.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philoxBlock(uint32_t key0, uint32_t key1, uint32_t block, uint64_t seed)
{
    uint32_t x0 = block, x1 = (uint32_t)seed, x2 = (uint32_t)(seed >> 32), x3 = 0, k0 = key0, k1 = key1;
#pragma unroll
    for (int r = 0; r < 10; r++)
    {
        const uint32_t hi0 = __umulhi(0xD2511F53u, x0), lo0 = 0xD2511F53u * x0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, x2), lo1 = 0xCD9E8D57u * x2;
        const uint32_t n0 = hi1 ^ x1 ^ k0, n2 = hi0 ^ x3 ^ k1;
        x0 = n0; x1 = lo1; x2 = n2; x3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(x0, x1, x2, x3);
}
__device__ __forceinline__ float uniform01(uint32_t v) { return (float)(v >> 8) * (1.0f / 16777216.0f); }

} // namespace rtb
