// rtb_bvh.h -- node test of the triangle-mesh hierarchy (RTB_PRIM_MESH).  Plain C++ (host + device): tests/bvh_bound_check.cpp
// compiles it for the host and checks the bound below on random pairs the reference's test accepts.
//
// A mesh must return the hit the run of the same triangles returns (include/rtb.h: RTB_PRIM_MESH).  So a node may be
// skipped only when no triangle below it can be ACCEPTED by the reference's test (rtb_device.cuh: triIntersectT) with
// t_ref <= best.  The reference's t_ref is not the geometric distance; this header bounds the difference.
//
// Notation as in rtb_pretest.h: float inputs e1 = a - b, e2 = a - c, d, b' = fl(a - o); exact determinants DetX of those
// floats; the reference's values detX_r with |detX_r - DetX| <= gamma_7 S_X, S_M <= dmx A1, S_B, S_G <= dmx bn E,
// S_T <= bn A1 (bn = |b'|_1, dmx = max |d_i|, A1 and E the per-triangle sums of rtb_pretest.h).
//
// Residual.  Cramer's identity DetB e1 + DetG e2 + DetT d = DetM b' holds exactly.  With the reference's determinants and
// the real quotients beta' = detB_r / detM_r, gamma', t' it leaves
//      o' + t' d = P' + R,   P' = a - beta' e1 - gamma' e2,   o' = a - b',
//      |R_i| <= (|eps_B| |e1_i| + |eps_G| |e2_i| + |eps_T| |d_i| + |eps_M| |b'_i|) / |detM_r|
//            <= 2 gamma_7 dmx bn (E^2 + A1) / |detM_r|  <=  kappa_g bn / |detM_r|,
//      kappa_g = RTB_PRE_EPS dmx (A1 + E^2)                          (RTB_PRE_EPS = 2^-19 >= 2 gamma_7).
// GRAZING BAND: |detM_r| <= RTB_BVH_C kappa_g.  Outside it |R_i| < bn / C.  Inside it the ray lies almost in the triangle's
// plane (|detM_r| / (dmx (A1 + E^2)) <= C 2^-19 ~ 0.002: a fraction of a degree for a well-shaped triangle; always for a
// sliver or zero-area facet) and the reference's t is rounding noise: the hierarchy does not promise to reproduce it.
//
// Accepted pair outside the band:
//   * P' is in the leaf box.  beta_r, gamma_r, 1 - beta_r - gamma_r >= -1e-4 (Triangle.cpp:102, 108) and the three weights
//     of P' over (a, a - e1, a - e2) sum to 1, so every coordinate of P' lies within 2 * 1.0001e-4 of the vertex extent
//     (plus the float roundings of the quotients, of alpha and of e1, e2, each below 2^-23 relative): leaf boxes are the
//     triangle's box widened on each side by RTB_BVH_SLACK times its extent on that axis, rounded outward.
//   * The ray point o + t' d is within |R_i| + |o_i - o'_i| < bn (1 / C + 2^-24) of P' on each axis; bn <= (1 + 2^-24) D,
//     D = the largest L1 distance from the origin to a point of the node's box.  So the slab interval of the node's box
//     widened by D * RTB_BVH_K (+ RTB_BVH_ABS times the box coordinates for the roundings of the widened planes) contains
//     t' -- after widening the computed interval by RTB_BVH_REL relative (quotient, subtraction, reciprocal; and
//     t_ref = fl(t') is within 2^-24 relative of t').
//   * t_ref >= 0.0005 (Triangle.cpp:90) implies t' >= RTB_BVH_TMIN.
// A node is therefore skipped only when the widened interval misses [RTB_BVH_TMIN, best].  An axis with d_i == 0 keeps the
// ray's coordinate exactly, so it skips the node when o_i is outside the widened slab and constrains nothing otherwise; an
// axis whose reciprocal is not finite (|d_i| < 2^-126) constrains nothing: neither produces inf - inf or 0 * inf.
#pragma once
#include <math.h>
#include <float.h>

#if defined(__CUDACC__)
#define RTB_BVH_FN __host__ __device__ __forceinline__
#else
#define RTB_BVH_FN inline
#endif

namespace rtb_bvh {

#define RTB_BVH_C 1024.0f                    // grazing band |detM_r| <= C kappa_g
#define RTB_BVH_SLACK 2.1e-4f                // leaf box widening per side, times the triangle's extent (>= 2 * 1.0001e-4 + roundings)
#define RTB_BVH_K 9.79e-4f                   // >= (1 / C + 2^-24)(1 + 2^-24)(1 + 4 * 2^-24): D -> slab widening
#define RTB_BVH_ABS 2.384185791015625e-07f   // 2^-22: roundings of lo - r, hi + r
#define RTB_BVH_REL 9.5367431640625e-07f     // 2^-20: relative widening of the computed interval
#define RTB_BVH_TMIN 4.9995e-4f              // t_ref >= 0.0005 => t' >= this
#define RTB_BVH_STACK 64                     // 62-bit keys: inner depth <= 62, one pending sibling per level

// one triangle's leaf box, from its vertices (9 floats a, b, c)
RTB_BVH_FN void leafBox(const float *v, float lo[3], float hi[3])
{
    for (int i = 0; i < 3; i++)
    {
        const float mn = fminf(fminf(v[i], v[3 + i]), v[6 + i]), mx = fmaxf(fmaxf(v[i], v[3 + i]), v[6 + i]);
        const float w = (mx - mn) * RTB_BVH_SLACK;
        lo[i] = nextafterf(mn - w, -INFINITY);
        hi[i] = nextafterf(mx + w, INFINITY);
    }
}

// per-ray constants; mode 0: finite reciprocal, 1: d_i == 0, 2: no constraint from this axis
struct Ray
{
    float o[3], inv[3];
    int mode[3];
};
RTB_BVH_FN Ray makeRay(float ox, float oy, float oz, float dx, float dy, float dz)
{
    Ray r;
    const float o[3] = {ox, oy, oz}, d[3] = {dx, dy, dz};
    for (int i = 0; i < 3; i++)
    {
        r.o[i] = o[i];
        r.inv[i] = 1.0f / d[i];
        r.mode[i] = d[i] == 0.0f ? 1 : (fabsf(r.inv[i]) <= FLT_MAX ? 0 : 2);
        if (r.mode[i] != 0) r.inv[i] = 0.0f;
    }
    return r;
}

// true: the node with box [lo, hi] may hold a triangle the reference accepts with t_ref <= best (visit it)
RTB_BVH_FN bool nodeHit(const Ray &r, const float lo[3], const float hi[3], float best)
{
    float D = 0.0f;
    for (int i = 0; i < 3; i++) D += fmaxf(fabsf(lo[i] - r.o[i]), fabsf(hi[i] - r.o[i]));
    const float wD = D * RTB_BVH_K;
    float tn = -INFINITY, tf = INFINITY;
    bool outside = false;
    for (int i = 0; i < 3; i++)
    {
        const float w = wD + (fabsf(lo[i]) + fabsf(hi[i])) * RTB_BVH_ABS;
        const float l = lo[i] - w, h = hi[i] + w;
        if (r.mode[i] == 0)
        {
            const float t0 = (l - r.o[i]) * r.inv[i], t1 = (h - r.o[i]) * r.inv[i];
            tn = fmaxf(tn, fminf(t0, t1));
            tf = fminf(tf, fmaxf(t0, t1));
        }
        else if (r.mode[i] == 1) outside = outside || !(r.o[i] >= l && r.o[i] <= h);
    }
    tn = tn - fabsf(tn) * RTB_BVH_REL;
    tf = tf + fabsf(tf) * RTB_BVH_REL;
    return !outside && tn <= tf && tf >= RTB_BVH_TMIN && tn <= best;
}

} // namespace rtb_bvh
