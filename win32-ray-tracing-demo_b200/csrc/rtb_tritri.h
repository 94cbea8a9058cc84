// rtb_tritri.h -- the exact triangle-triangle overlap test of the triangle queries (rtb_query_triangles, DESIGN 3g).  Plain C++
// (host + device), under the rules of rtb_closest.h: tests/tritri_check.cpp compiles it for the host with -ffp-contract=off, the
// library with -fmad=false, and only + - * and comparisons are used (no fma).
//
// Contract: intersect(p, q) is true exactly when the two closed triangles p, q (9 floats each: three vertices) share a point in
// exact real arithmetic -- touching counts -- unless either is DEGENERATE: a non-finite coordinate, or three exactly collinear
// vertices (repeated vertices included).  Degenerate triangles intersect nothing.
//
// Predicates.  orient3d(a, b, c, d) = det[a - d; b - d; c - d] and orient2d(a, b, c) = det[a - c; b - c] of float points, in
// double, with Shewchuk's forward error bounds as the filter ("Adaptive Precision Floating-Point Arithmetic and Fast Robust
// Geometric Predicates", 1997: o3derrboundA, ccwerrboundA).  When the filter cannot decide, the same determinant is evaluated
// exactly: as the cofactor expansion of the 4x4 (3x3) determinant with a column of ones, a sum of 24 (6) signed products of
// three (two) input floats.  A product of two floats is exact in double (24 + 24 <= 53 bits); a third factor makes it one
// Two-Product (Dekker split), two doubles whose sum is exact; the terms are summed by Grow-Expansion (Two-Sum) into a
// nonoverlapping expansion whose largest component carries the sign.  Inputs are floats, so nothing overflows or underflows:
// a product of three floats lies in [2^-447, 2^384] or is 0, Two-Product's error term is far above 2^-1022, and the filter's
// differences (<= 2^129) and their cubes (< 2^388) stay in range, which is the condition of Shewchuk's bounds.  So every sign
// is exact for every finite float input, and the host and the device agree because the decisions are exact, not because their
// bits match.  RTB_TRITRI_COUNT(k), when defined, is called on each exact evaluation (k = 3 or 2): the host check counts them.
//
// Algorithm: Guigue and Devillers, "Fast and Robust Triangle-Triangle Overlap Test Using Orientation Predicates" (Journal of
// Graphics Tools 8(1), 2003): the signs of p's vertices against q's plane and of q's against p's, the early exits when one
// triangle lies strictly on one side, the canonical permutation, then two orient3d interval predicates.  A coplanar pair is
// decided in the axis plane in which p's projection has a nonzero orient2d (exact, and one exists for a non-degenerate p;
// projecting the common plane onto it is an affine bijection, so the answer is the planar one): two closed triangles overlap
// exactly when an edge of one meets an edge of the other, or a vertex of one lies in the other, from 18 orient2d signs.
//
// Pruning: boxesOverlap tests closed boxes.  A shared point lies in both triangles' boxes, so a node whose box is strictly
// separated from the query's on one axis holds no intersecting triangle when it contains its triangles' vertices a, fl(a - e1),
// fl(a - e2) -- which DESIGN 3e proves for every node after a build and after a refit.
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define RTB_TRITRI_FN __host__ __device__ __forceinline__
#define RTB_TRITRI_SLOW __host__ __device__ __noinline__
#define RTB_TRITRI_CALL __host__ __device__ __noinline__ // a call of its own: a walk that calls it keeps its own registers
#else
#define RTB_TRITRI_FN inline
#define RTB_TRITRI_SLOW inline
#define RTB_TRITRI_CALL inline
#endif
#ifndef RTB_TRITRI_COUNT
#define RTB_TRITRI_COUNT(k)
#endif

namespace rtb_tritri {

// ---- expansion arithmetic (Shewchuk 1997) -----------------------------------------------------------------------------------
RTB_TRITRI_FN void twoSum(double a, double b, double &x, double &y)
{
    x = a + b;
    const double bv = x - a, av = x - bv;
    y = (a - av) + (b - bv);
}

RTB_TRITRI_FN void split(double a, double &hi, double &lo)
{
    const double c = 134217729.0 * a; // 2^27 + 1
    hi = c - (c - a);
    lo = a - hi;
}

RTB_TRITRI_FN void twoProduct(double a, double b, double &x, double &y)
{
    x = a * b;
    double ah, al, bh, bl;
    split(a, ah, al);
    split(b, bh, bl);
    y = al * bl - (((x - ah * bh) - al * bh) - ah * bl);
}

// e[0 .. n) += b, zero components dropped; in place (Grow-Expansion); returns the new length
RTB_TRITRI_FN int grow(double *e, int n, double b)
{
    double q = b;
    int m = 0;
    for (int i = 0; i < n; i++)
    {
        double h;
        twoSum(q, e[i], q, h);
        if (h != 0.0) e[m++] = h;
    }
    if (q != 0.0 || m == 0) e[m++] = q;
    return m;
}

RTB_TRITRI_FN int signOf(double x) { return (x > 0.0) - (x < 0.0); }

// exact sign of det[a - d; b - d; c - d]: det4 [[a, 1], [b, 1], [c, 1], [d, 1]] = -|bcd| + |acd| - |abd| + |abc|
RTB_TRITRI_SLOW int orient3dExact(const float *a, const float *b, const float *c, const float *d)
{
    RTB_TRITRI_COUNT(3);
    const float *rows[4][3] = {{b, c, d}, {a, c, d}, {a, b, d}, {a, b, c}};
    double e[48];
    int n = 0;
    for (int r = 0; r < 4; r++)
    {
        const float *p = rows[r][0], *q = rows[r][1], *s = rows[r][2];
        const double sg = (r & 1) ? 1.0 : -1.0;
        // |p q s| = px qy sz - px qz sy - py qx sz + py qz sx + pz qx sy - pz qy sx
        const int i0[6] = {0, 0, 1, 1, 2, 2}, i1[6] = {1, 2, 0, 2, 0, 1}, i2[6] = {2, 1, 2, 0, 1, 0};
        for (int t = 0; t < 6; t++)
        {
            const double m = (double)p[i0[t]] * (double)q[i1[t]]; // exact
            double x, y;
            twoProduct(m, (double)s[i2[t]], x, y);
            const double g = (t == 0 || t == 3 || t == 4) ? sg : -sg;
            n = grow(e, n, g * y);
            n = grow(e, n, g * x);
        }
    }
    return signOf(e[n - 1]);
}

// exact sign of det[a - c; b - c] over the axes (u, v): ax by - ay bx - ax cy + ay cx + bx cy - by cx
RTB_TRITRI_SLOW int orient2dExact(const float *a, const float *b, const float *c, int u, int v)
{
    RTB_TRITRI_COUNT(2);
    const double t[6] = {(double)a[u] * b[v], -((double)a[v] * b[u]), -((double)a[u] * c[v]), (double)a[v] * c[u],
                         (double)b[u] * c[v], -((double)b[v] * c[u])}; // each product exact
    double e[6];
    int n = 0;
    for (int i = 0; i < 6; i++) n = grow(e, n, t[i]);
    return signOf(e[n - 1]);
}

// ---- filtered predicates ----------------------------------------------------------------------------------------------------
#define RTB_TRITRI_EPS 1.1102230246251565e-16 // 2^-53
RTB_TRITRI_FN int orient3d(const float *a, const float *b, const float *c, const float *d)
{
    const double adx = (double)a[0] - d[0], ady = (double)a[1] - d[1], adz = (double)a[2] - d[2];
    const double bdx = (double)b[0] - d[0], bdy = (double)b[1] - d[1], bdz = (double)b[2] - d[2];
    const double cdx = (double)c[0] - d[0], cdy = (double)c[1] - d[1], cdz = (double)c[2] - d[2];
    const double bc = bdx * cdy, cb = cdx * bdy, ca = cdx * ady, ac = adx * cdy, ab = adx * bdy, ba = bdx * ady;
    const double det = adz * (bc - cb) + bdz * (ca - ac) + cdz * (ab - ba);
    const double perm = (fabs(bc) + fabs(cb)) * fabs(adz) + (fabs(ca) + fabs(ac)) * fabs(bdz) + (fabs(ab) + fabs(ba)) * fabs(cdz);
    const double bound = (7.0 + 56.0 * RTB_TRITRI_EPS) * RTB_TRITRI_EPS * perm;
    if (det > bound || -det > bound) return signOf(det);
    return orient3dExact(a, b, c, d);
}

// orient2d of the projections onto the axes (u, v)
RTB_TRITRI_FN int orient2d(const float *a, const float *b, const float *c, int u, int v)
{
    const double l = ((double)a[u] - c[u]) * ((double)b[v] - c[v]), r = ((double)a[v] - c[v]) * ((double)b[u] - c[u]);
    const double det = l - r;
    // a factor that is 0 in double is 0 exactly (distinct floats differ in double), so a zero or sign-opposed side decides
    if (l == 0.0 || r == 0.0 || (l > 0.0) != (r > 0.0)) return signOf(det);
    const double bound = (3.0 + 16.0 * RTB_TRITRI_EPS) * RTB_TRITRI_EPS * (fabs(l) + fabs(r));
    if (det > bound || -det > bound) return signOf(det);
    return orient2dExact(a, b, c, u, v);
}

// ---- triangles --------------------------------------------------------------------------------------------------------------
RTB_TRITRI_FN bool finite3(const float *v) { return fabsf(v[0]) <= 3.40282347e38f && fabsf(v[1]) <= 3.40282347e38f && fabsf(v[2]) <= 3.40282347e38f; }

// a non-finite coordinate, or all three axis projections of zero area (collinear or repeated vertices)
RTB_TRITRI_FN bool degenerate(const float *t)
{
    if (!(finite3(t) && finite3(t + 3) && finite3(t + 6))) return true;
    return orient2d(t, t + 3, t + 6, 0, 1) == 0 && orient2d(t, t + 3, t + 6, 1, 2) == 0 && orient2d(t, t + 3, t + 6, 2, 0) == 0;
}

RTB_TRITRI_FN void box(const float *t, float lo[3], float hi[3])
{
    for (int i = 0; i < 3; i++)
    {
        lo[i] = t[i] < t[3 + i] ? t[i] : t[3 + i];
        lo[i] = t[6 + i] < lo[i] ? t[6 + i] : lo[i];
        hi[i] = t[i] > t[3 + i] ? t[i] : t[3 + i];
        hi[i] = t[6 + i] > hi[i] ? t[6 + i] : hi[i];
    }
}

// closed boxes: false only when an axis strictly separates them
RTB_TRITRI_FN bool boxesOverlap(const float lo[3], const float hi[3], const float lo2[3], const float hi2[3])
{
    return !(hi[0] < lo2[0] || hi2[0] < lo[0] || hi[1] < lo2[1] || hi2[1] < lo[1] || hi[2] < lo2[2] || hi2[2] < lo[2]);
}

// Coplanar pair, projected onto (u, v) where p's projection has orientation sp != 0 (q's then has one too).
RTB_TRITRI_FN bool overlap2d(const float *p, const float *q, int u, int v, int sp)
{
    const float *P[3] = {p, p + 3, p + 6}, *Q[3] = {q, q + 3, q + 6};
    const int sq = orient2d(Q[0], Q[1], Q[2], u, v);
    int op[3][3], oq[3][3]; // op[e][j]: q's vertex j against p's edge e (P[e] -> P[e + 1]); oq[e][j] likewise
    for (int e = 0; e < 3; e++)
        for (int j = 0; j < 3; j++)
        {
            op[e][j] = orient2d(P[e], P[(e + 1) % 3], Q[j], u, v);
            oq[e][j] = orient2d(Q[e], Q[(e + 1) % 3], P[j], u, v);
        }
    for (int j = 0; j < 3; j++) // a vertex of one inside the other, boundary included
    {
        if (op[0][j] * sp >= 0 && op[1][j] * sp >= 0 && op[2][j] * sp >= 0) return true;
        if (oq[0][j] * sq >= 0 && oq[1][j] * sq >= 0 && oq[2][j] * sq >= 0) return true;
    }
    // edges that cross or touch without being collinear (collinear overlapping edges put a vertex on the other's boundary)
    for (int e = 0; e < 3; e++)
        for (int f = 0; f < 3; f++)
        {
            const int a0 = op[e][f], a1 = op[e][(f + 1) % 3], b0 = oq[f][e], b1 = oq[f][(e + 1) % 3];
            if (a0 * a1 <= 0 && b0 * b1 <= 0 && (a0 != 0 || a1 != 0)) return true;
        }
    return false;
}

RTB_TRITRI_FN bool coplanar(const float *p, const float *q)
{
    for (int ax = 0; ax < 3; ax++)
    {
        const int u = (ax + 1) % 3, v = (ax + 2) % 3;
        const int sp = orient2d(p, p + 3, p + 6, u, v);
        if (sp != 0) return overlap2d(p, q, u, v, sp);
    }
    return false; // p degenerate: not reached for the inputs intersect() passes on
}

// Guigue-Devillers' interval test of the canonical form: p1 alone on its side of q's plane, q's vertices ordered so that
// p1 sees q1 q2 q3 counterclockwise
RTB_TRITRI_FN bool minMax(const float *p1, const float *q1, const float *r1, const float *p2, const float *q2, const float *r2)
{
    if (orient3d(p2, p1, q2, q1) > 0) return false;
    return !(orient3d(p2, r1, r2, p1) > 0);
}

RTB_TRITRI_FN bool canonical2(const float *p1, const float *q1, const float *r1, const float *p2, const float *q2, const float *r2,
                              int dp2, int dq2, int dr2)
{
    if (dp2 > 0)
    {
        if (dq2 > 0) return minMax(p1, r1, q1, r2, p2, q2);
        if (dr2 > 0) return minMax(p1, r1, q1, q2, r2, p2);
        return minMax(p1, q1, r1, p2, q2, r2);
    }
    if (dp2 < 0)
    {
        if (dq2 < 0) return minMax(p1, q1, r1, r2, p2, q2);
        if (dr2 < 0) return minMax(p1, q1, r1, q2, r2, p2);
        return minMax(p1, r1, q1, p2, q2, r2);
    }
    if (dq2 < 0)
    {
        if (dr2 >= 0) return minMax(p1, r1, q1, q2, r2, p2);
        return minMax(p1, q1, r1, p2, q2, r2);
    }
    if (dq2 > 0)
    {
        if (dr2 > 0) return minMax(p1, r1, q1, p2, q2, r2);
        return minMax(p1, q1, r1, q2, r2, p2);
    }
    if (dr2 > 0) return minMax(p1, q1, r1, r2, p2, q2);
    return minMax(p1, r1, q1, r2, p2, q2); // dr2 < 0: all three zero is the coplanar case, handled before
}

// The exact test of two triangles that are not degenerate (the caller checks: degenerate() of each)
RTB_TRITRI_FN bool intersectValid(const float *p, const float *q)
{
    const float *p1 = p, *q1 = p + 3, *r1 = p + 6, *p2 = q, *q2 = q + 3, *r2 = q + 6;
    const int dp1 = orient3d(p2, q2, p1, r2), dq1 = orient3d(p2, q2, q1, r2), dr1 = orient3d(p2, q2, r1, r2);
    if (dp1 * dq1 > 0 && dp1 * dr1 > 0) return false;
    const int dp2 = orient3d(p1, q1, p2, r1), dq2 = orient3d(p1, q1, q2, r1), dr2 = orient3d(p1, q1, r2, r1);
    if (dp2 * dq2 > 0 && dp2 * dr2 > 0) return false;
    if (dp1 > 0)
    {
        if (dq1 > 0) return canonical2(r1, p1, q1, p2, r2, q2, dp2, dr2, dq2);
        if (dr1 > 0) return canonical2(q1, r1, p1, p2, r2, q2, dp2, dr2, dq2);
        return canonical2(p1, q1, r1, p2, q2, r2, dp2, dq2, dr2);
    }
    if (dp1 < 0)
    {
        if (dq1 < 0) return canonical2(r1, p1, q1, p2, q2, r2, dp2, dq2, dr2);
        if (dr1 < 0) return canonical2(q1, r1, p1, p2, q2, r2, dp2, dq2, dr2);
        return canonical2(p1, q1, r1, p2, r2, q2, dp2, dr2, dq2);
    }
    if (dq1 < 0)
    {
        if (dr1 >= 0) return canonical2(q1, r1, p1, p2, r2, q2, dp2, dr2, dq2);
        return canonical2(p1, q1, r1, p2, q2, r2, dp2, dq2, dr2);
    }
    if (dq1 > 0)
    {
        if (dr1 > 0) return canonical2(p1, q1, r1, p2, r2, q2, dp2, dr2, dq2);
        return canonical2(q1, r1, p1, p2, q2, r2, dp2, dq2, dr2);
    }
    if (dr1 > 0) return canonical2(r1, p1, q1, p2, q2, r2, dp2, dq2, dr2);
    if (dr1 < 0) return canonical2(r1, p1, q1, p2, r2, q2, dp2, dr2, dq2);
    return coplanar(p, q);
}

// q's degeneracy test and the exact test, for a p already known not to be degenerate (the query side of a walk)
RTB_TRITRI_CALL bool meets(const float *p, const float *q) { return !degenerate(q) && intersectValid(p, q); }

RTB_TRITRI_FN bool intersect(const float *p, const float *q) { return !degenerate(p) && meets(p, q); }

} // namespace rtb_tritri
