// rtb_winding.h -- signed solid angles and first-order moments of triangles: the generalised winding number of the winding
// queries (rtb_query_winding, DESIGN 3f).  Plain C++ (host + device), like rtb_closest.h: tests/winding_check.cpp compiles it
// for the host with -ffp-contract=off, the library with -fmad=false, and only + - * /, sqrtf and comparisons are used, so
// both evaluate every expression below in the same float32 operations and return the same bits.
//
// Winding number (Barill et al., "Fast Winding Numbers for Soups and Clouds", SIGGRAPH 2018): w(p) = sum_t Omega_t(p) / 4 pi.
// For a closed, consistently oriented surface it is 1 inside and 0 outside (-1 inside when the facets face inwards); an open
// or imperfect soup gives fractional values that degrade gracefully.
//
// Input: the packed triangle record of DScene::loose / mesh_tris, t = {a.xyz, e1.xyz, e2.xyz, n.xyz}, e1 = a - b, e2 = a - c.
// The vertices used are a, b' = fl(a + ab), c' = fl(a + ac) with ab = -e1, ac = -e2, exactly as rtb_closest.h reconstructs
// them.  Orientation comes from the vertex order (right-hand rule: (b - a) x (c - a) = e1 x e2 points outwards), never from
// the stored normal n.
//
// Accuracy (tests/winding_check.cpp, against float64 on the same float vertices; eps = 2^-24):
//   * atan2: |atan2(y, x) - atan2_64(y, x)| <= RTB_ATAN2_REL |atan2_64(y, x)| for all finite and infinite y, x, signed
//     zeros included (IEEE special cases; NaN in, NaN out).  The polynomial alone is within 1.6e-8 relative of atan on [0, 1].
//   * solidAngle: with A, B, C as below, D = hypot(det, den) of the float64 values and L = |A| |B| |C|:
//     |Omega - Omega_64| <= RTB_SOLID_ABS + RTB_SOLID_COND L / D, modulo 4 pi.  L / D grows only near the triangle's edges
//     (D vanishes when p lies on an edge); modulo 4 pi because a point in the triangle's plane inside it sees +-2 pi,
//     whichever sign its rounded det takes.  A point on a vertex (det = den = 0) contributes 0.
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define RTB_WINDING_FN __host__ __device__ __forceinline__
#else
#define RTB_WINDING_FN inline
#endif

namespace rtb_winding {

#define RTB_WINDING_PI 3.14159274101257324f     // fl(pi)
#define RTB_WINDING_PI_2 1.57079637050628662f   // fl(pi / 2)
#define RTB_WINDING_INV4PI 0.0795774715459476679f // fl(1 / (4 pi))
#define RTB_ATAN2_REL 2.4e-7f                   // stated relative bound of atan2 (measured worst: tests/winding_check.cpp)
#define RTB_SOLID_ABS 1.0e-6f                   // stated absolute part of the solidAngle bound (radians)
#define RTB_SOLID_COND 2.0e-6f                  // stated conditioning part of the solidAngle bound (times L / D)

// atan(t) = t P(t^2) on [0, 1]: minimax in relative error (Lawson iterations), degree 8 in t^2, coefficients rounded to float
RTB_WINDING_FN float atanUnit(float t)
{
    const float s = t * t;
    float q = 0.0028498906176537275f;
    q = q * s + -0.016068633645772934f;
    q = q * s + 0.04269153252243996f;
    q = q * s + -0.0750429555773735f;
    q = q * s + 0.10640934854745865f;
    q = q * s + -0.14203645288944244f;
    q = q * s + 0.1999261975288391f;
    q = q * s + -0.3333307206630707f;
    q = q * s + 1.0f;
    return t * q;
}

// x < 0, or x is -0 (1 / -0 = -inf)
RTB_WINDING_FN bool negative(float x) { return x < 0.0f || (x == 0.0f && 1.0f / x < 0.0f); }

// atan2 by range reduction to [0, 1] and atanUnit: libm's and CUDA's atan2f differ in their last bits, this does not
RTB_WINDING_FN float atan2(float y, float x)
{
    if (x != x || y != y) return x + y;
    const float ax = negative(x) ? -x : x, ay = negative(y) ? -y : y; // +0 for -0, so the signs below come from x and y alone
    const bool swap = ay > ax;
    const float mx = swap ? ay : ax, mn = swap ? ax : ay;
    // mn / mx in [0, 1]: 0 / 0 -> 0 (the signed-zero cases), inf / inf -> 1 (the diagonal)
    const float t = mx > 0.0f ? (mn == mx ? 1.0f : mn / mx) : 0.0f;
    float r = atanUnit(t);
    if (swap) r = RTB_WINDING_PI_2 - r;
    if (negative(x)) r = RTB_WINDING_PI - r;
    return negative(y) ? -r : r;
}

RTB_WINDING_FN float dot3(const float u[3], const float v[3]) { return u[0] * v[0] + u[1] * v[1] + u[2] * v[2]; }
RTB_WINDING_FN float norm3(const float u[3]) { return sqrtf(dot3(u, u)); }

// signed solid angle of the packed triangle t (12 floats) seen from p, by van Oosterom and Strackee (IEEE Trans. Biomed.
// Eng. 30(2), 1983): Omega = 2 atan2(det[A B C], |A||B||C| + (A.B)|C| + (A.C)|B| + (B.C)|A|), A = a - p, B = b' - p, C = c' - p
RTB_WINDING_FN float solidAngle(const float p[3], const float *t)
{
    const float A[3] = {t[0] - p[0], t[1] - p[1], t[2] - p[2]};
    const float B[3] = {(t[0] + -t[3]) - p[0], (t[1] + -t[4]) - p[1], (t[2] + -t[5]) - p[2]};
    const float Cv[3] = {(t[0] + -t[6]) - p[0], (t[1] + -t[7]) - p[1], (t[2] + -t[8]) - p[2]};
    const float bc[3] = {B[1] * Cv[2] - B[2] * Cv[1], B[2] * Cv[0] - B[0] * Cv[2], B[0] * Cv[1] - B[1] * Cv[0]};
    const float det = dot3(A, bc);
    const float la = norm3(A), lb = norm3(B), lc = norm3(Cv);
    const float den = la * lb * lc + dot3(A, B) * lc + dot3(A, Cv) * lb + dot3(B, Cv) * la;
    if (det == 0.0f && den == 0.0f) return 0.0f; // p on a vertex
    return 2.0f * rtb_winding::atan2(det, den);
}

// first-order moments of the packed triangle t: area vector N = (e1 x e2) / 2, centroid c, and r >= the largest distance
// from c to a vertex (rounded outward)
RTB_WINDING_FN void triMoment(const float *t, float N[3], float c[3], float &r)
{
    const float a[3] = {t[0], t[1], t[2]};
    const float b[3] = {t[0] + -t[3], t[1] + -t[4], t[2] + -t[5]}, cc[3] = {t[0] + -t[6], t[1] + -t[7], t[2] + -t[8]};
    N[0] = (t[4] * t[8] - t[5] * t[7]) * 0.5f;
    N[1] = (t[5] * t[6] - t[3] * t[8]) * 0.5f;
    N[2] = (t[3] * t[7] - t[4] * t[6]) * 0.5f;
    for (int i = 0; i < 3; i++) c[i] = (a[i] + b[i] + cc[i]) * (1.0f / 3.0f);
    const float da[3] = {a[0] - c[0], a[1] - c[1], a[2] - c[2]};
    const float db[3] = {b[0] - c[0], b[1] - c[1], b[2] - c[2]};
    const float dc[3] = {cc[0] - c[0], cc[1] - c[1], cc[2] - c[2]};
    float m = dot3(da, da), e = dot3(db, db);
    m = e > m ? e : m;
    e = dot3(dc, dc);
    m = e > m ? e : m;
    r = sqrtf(m) * 1.00000095367431641f; // (1 + 2^-20): outward over the roundings of the centroid and the distances
}

// the first-order far-field term of a cluster with area vector N and centre c, in winding-number units:
// N . (c - p) / (4 pi |c - p|^3)
RTB_WINDING_FN float dipole(const float p[3], const float N[3], const float c[3])
{
    const float d[3] = {c[0] - p[0], c[1] - p[1], c[2] - p[2]};
    const float d2 = dot3(d, d);
    const float l = sqrtf(d2);
    return dot3(N, d) / (d2 * l) * RTB_WINDING_INV4PI;
}

// true: p lies farther than beta r from c, so the cluster's dipole stands for it (beta = +inf: never; r = 0 and beta = inf
// give NaN, which is not far either)
RTB_WINDING_FN bool far(const float p[3], const float c[3], float r, float beta)
{
    const float d[3] = {c[0] - p[0], c[1] - p[1], c[2] - p[2]};
    const float br = beta * r;
    return dot3(d, d) > br * br;
}

} // namespace rtb_winding
