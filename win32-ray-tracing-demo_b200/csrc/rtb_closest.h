// rtb_closest.h -- closest point on a triangle and the squared distances of the point queries (rtb_query_points).  Plain C++
// (host + device): tests/closest_point_check.cpp compiles it for the host with -ffp-contract=off, the library with -fmad=false,
// so both evaluate every expression below in the same float32 operations and return the same bits.  Only + - * /, sqrtf and
// comparisons are used (no fmaf; no fminf / fmaxf either, whose result for +0 / -0 is not fixed across platforms).
//
// Input: the packed triangle record of DScene::loose / mesh_tris, t = {a.xyz, e1.xyz, e2.xyz, n.xyz}, e1 = a - b, e2 = a - c.
// The vertices used are a, b' = fl(a + ab), c' = fl(a + ac) with ab = -e1, ac = -e2 (negation is exact).
//
// Closest point: Ericson, Real-Time Collision Detection, 5.1.5 (Voronoi regions of a, b', ab, c', ac, b'c', then the interior),
// in the operation order written below.  The sub-triangle areas va, vb, vc take the book's cross-product form
// n . ((x - p) x (y - p)), n = ab x ac, and the interior point is the projection of p onto the plane: on thin triangles both
// are far better conditioned than the Lagrange-identity form d1 d4 - d3 d2 and the barycentric quotient, whose float error
// grows as 1 / sin^2 of the triangle's angle (a relative distance error of 0.7 was seen on collinear float triangles).
// DEGENERATE triangles -- zero area, collinear, slivers: n . n not finite, or not above 2^-24 |ab|^2 |ac|^2 (sin^2 of the angle
// at a) -- take the nearest of the three edges ab, ac, b'c', each a segment with its parameter clamped to [0, 1] (NaN -> 0);
// ties go to the first.  Finally q is clamped per axis into [min, max] of a_i, b'_i, c'_i (a NaN coordinate becomes the min):
// q is finite whenever the vertices are.  Accuracy (tests/closest_point_check.cpp, against float64 on the same vertices):
// |sqrt(d2) - d| <= 1e-4 (|p - a| + extent) + 8 ulp of the largest coordinate (the worst seen is 2.4e-5).
//
// Pruning (why a BVH walk returns the linear scan's answer bit for bit).  d2 = fl(fl(fl(dx dx) + fl(dy dy)) + fl(dz dz)),
// dx = fl(p_x - q_x); boxDist2 evaluates the same expression with the per-axis gap lo_i - p_i, p_i - hi_i or 0.  When q_i lies in
// [lo_i, hi_i], |p_i - q_i| >= gap_i exactly, and round-to-nearest is monotone, so every later operation keeps the order:
// boxDist2(p, box) <= d2 in float.  q lies in [min, max] of a, b', c', which lies inside rtb_bvh::leafBox of the raw vertices
// (the leaf box is widened by RTB_BVH_SLACK of the extent plus one outward ulp, far more than the rounding of
// fl(a - fl(a - b)); tests/closest_point_check.cpp checks it), and inner boxes are unions of leaf boxes after a build and after
// a refit.  So a node with boxDist2 > best holds no triangle that can win, whatever the tree's shape.
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define RTB_CLOSEST_FN __host__ __device__ __forceinline__
#else
#define RTB_CLOSEST_FN inline
#endif

namespace rtb_closest {

#define RTB_CLOSEST_FLAT 5.9604644775390625e-08f // 2^-24: sin^2 of the triangle's angle at a below which it counts as degenerate

RTB_CLOSEST_FN float dot3(const float u[3], const float v[3]) { return u[0] * v[0] + u[1] * v[1] + u[2] * v[2]; }

// n . (u x v), with u = p - x and v = p - y: the n . ((x - p) x (y - p)) of Ericson's regions
RTB_CLOSEST_FN float triple(const float n[3], const float u[3], const float v[3])
{
    const float w[3] = {u[1] * v[2] - u[2] * v[1], u[2] * v[0] - u[0] * v[2], u[0] * v[1] - u[1] * v[0]};
    return dot3(n, w);
}

// squared distance in the fixed order of the contract
RTB_CLOSEST_FN float dist2(float dx, float dy, float dz) { return dx * dx + dy * dy + dz * dz; }

// segment parameter into [0, 1]; NaN -> 0
RTB_CLOSEST_FN float clamp01(float x) { return x > 0.0f ? (x < 1.0f ? x : 1.0f) : 0.0f; }

// squared distance from p to the box [lo, hi]
RTB_CLOSEST_FN float boxDist2(const float p[3], const float lo[3], const float hi[3])
{
    float g[3];
    for (int i = 0; i < 3; i++) g[i] = p[i] < lo[i] ? lo[i] - p[i] : (p[i] > hi[i] ? p[i] - hi[i] : 0.0f);
    return dist2(g[0], g[1], g[2]);
}

// q clamped into [lo, hi] (a NaN coordinate -> lo), and its squared distance from p
RTB_CLOSEST_FN float finish(const float p[3], const float lo[3], const float hi[3], float q[3])
{
    for (int i = 0; i < 3; i++)
    {
        if (!(q[i] >= lo[i])) q[i] = lo[i];
        if (q[i] > hi[i]) q[i] = hi[i];
    }
    return dist2(p[0] - q[0], p[1] - q[1], p[2] - q[2]);
}

// point s0 + d * clamp01(dot(p - s0, d) / dot(d, d)) of the segment from s0 along d
RTB_CLOSEST_FN void segmentPoint(const float p[3], const float s0[3], const float d[3], float q[3])
{
    const float sp[3] = {p[0] - s0[0], p[1] - s0[1], p[2] - s0[2]};
    const float s = clamp01(dot3(sp, d) / dot3(d, d));
    for (int i = 0; i < 3; i++) q[i] = s0[i] + d[i] * s;
}

// closest point q of the packed triangle t (12 floats) to p; returns its squared distance d2
RTB_CLOSEST_FN float closestPoint(const float p[3], const float *t, float q[3])
{
    const float a[3] = {t[0], t[1], t[2]};
    const float ab[3] = {-t[3], -t[4], -t[5]}, ac[3] = {-t[6], -t[7], -t[8]};
    const float b[3] = {a[0] + ab[0], a[1] + ab[1], a[2] + ab[2]}, c[3] = {a[0] + ac[0], a[1] + ac[1], a[2] + ac[2]};
    float lo[3], hi[3];
    for (int i = 0; i < 3; i++)
    {
        lo[i] = a[i] < b[i] ? a[i] : b[i];
        lo[i] = c[i] < lo[i] ? c[i] : lo[i];
        hi[i] = a[i] > b[i] ? a[i] : b[i];
        hi[i] = c[i] > hi[i] ? c[i] : hi[i];
    }
    const float ap[3] = {p[0] - a[0], p[1] - a[1], p[2] - a[2]};
    const float bp[3] = {p[0] - b[0], p[1] - b[1], p[2] - b[2]};
    const float cp[3] = {p[0] - c[0], p[1] - c[1], p[2] - c[2]};
    const float n[3] = {ab[1] * ac[2] - ab[2] * ac[1], ab[2] * ac[0] - ab[0] * ac[2], ab[0] * ac[1] - ab[1] * ac[0]};
    const float nn = dot3(n, n);
    if (!(nn > dot3(ab, ab) * dot3(ac, ac) * RTB_CLOSEST_FLAT && nn <= 3.40282347e38f))
    { // degenerate: the nearest of the edges ab, ac, b'c'
        const float bc[3] = {c[0] - b[0], c[1] - b[1], c[2] - b[2]};
        float r[3];
        segmentPoint(p, a, ab, q);
        float best = finish(p, lo, hi, q);
        segmentPoint(p, a, ac, r);
        float e = finish(p, lo, hi, r);
        if (e < best) { best = e; q[0] = r[0]; q[1] = r[1]; q[2] = r[2]; }
        segmentPoint(p, b, bc, r);
        e = finish(p, lo, hi, r);
        if (e < best) { best = e; q[0] = r[0]; q[1] = r[1]; q[2] = r[2]; }
        return best;
    }
    const float d1 = dot3(ab, ap), d2 = dot3(ac, ap);
    const float d3 = dot3(ab, bp), d4 = dot3(ac, bp);
    const float d5 = dot3(ab, cp), d6 = dot3(ac, cp);
    // signed areas of the sub-triangles in Ericson's cross-product form (better conditioned than d1 d4 - d3 d2 on thin triangles)
    const float vc = triple(n, ap, bp), vb = triple(n, cp, ap), va = triple(n, bp, cp);
    if (d1 <= 0.0f && d2 <= 0.0f)
    { // vertex a
        q[0] = a[0]; q[1] = a[1]; q[2] = a[2];
    }
    else if (d3 >= 0.0f && d4 <= d3)
    { // vertex b'
        q[0] = b[0]; q[1] = b[1]; q[2] = b[2];
    }
    else if (vc <= 0.0f && d1 >= 0.0f && d3 <= 0.0f)
    { // edge ab
        const float v = clamp01(d1 / (d1 - d3));
        for (int i = 0; i < 3; i++) q[i] = a[i] + ab[i] * v;
    }
    else if (d6 >= 0.0f && d5 <= d6)
    { // vertex c'
        q[0] = c[0]; q[1] = c[1]; q[2] = c[2];
    }
    else if (vb <= 0.0f && d2 >= 0.0f && d6 <= 0.0f)
    { // edge ac
        const float w = clamp01(d2 / (d2 - d6));
        for (int i = 0; i < 3; i++) q[i] = a[i] + ac[i] * w;
    }
    else if (va <= 0.0f && (d4 - d3) >= 0.0f && (d5 - d6) >= 0.0f)
    { // edge b'c'
        const float w = clamp01((d4 - d3) / ((d4 - d3) + (d5 - d6)));
        for (int i = 0; i < 3; i++) q[i] = b[i] + (c[i] - b[i]) * w;
    }
    else
    { // interior: the projection onto the plane
        const float h = dot3(ap, n) / nn;
        for (int i = 0; i < 3; i++) q[i] = p[i] - n[i] * h;
    }
    return finish(p, lo, hi, q);
}

} // namespace rtb_closest
