// CPU check of the point-query distance function (csrc/rtb_closest.h), compiled by tests/test_point_query.py with
// g++ -O2 -std=c++17 -ffp-contract=off.
//
// Draws seeded (point, triangle) pairs: random triangles, and adversarial ones -- slivers, zero-area and collinear triangles,
// repeated vertices, axis-flat triangles, coordinates offset up to 1e6 with extents down to 1e-6 -- with points near and far,
// on the vertices, on the edges and exactly in the triangle's plane.  Each triangle is packed as the library packs it
// (a, e1 = fl(a - b), e2 = fl(a - c), n).  For each pair it checks:
//   * q lies inside rtb_bvh::leafBox of the raw vertices (the containment the pruning rests on);
//   * boxDist2(p, leafBox) <= d2 (the pruning lemma itself);
//   * q and d2 are finite;
//   * |sqrt(d2) - dist64| <= TOL (|p - a| + extent) + ULPS ulp of the largest coordinate, dist64 = the float64 distance to the
//     triangle (a, b', c') the function works on (the float coordinates of p and q carry a rounding of their magnitude).
// usage: closest_point_check <seed> <pairs>; prints the counts and the largest relative error, exit status 1 on a violation.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <random>

#include "../win32-ray-tracing-demo_b200/csrc/rtb_bvh.h"
#include "../win32-ray-tracing-demo_b200/csrc/rtb_closest.h"

static const double TOL = 1e-4, ULPS = 8;

struct D3 { double x, y, z; };
static D3 sub(D3 a, D3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
static D3 add(D3 a, D3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
static D3 mul(D3 a, double s) { return {a.x * s, a.y * s, a.z * s}; }
static double dot(D3 a, D3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static D3 cross(D3 a, D3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }

static double segDist(D3 p, D3 s0, D3 s1)
{
    const D3 d = sub(s1, s0);
    const double dd = dot(d, d);
    double t = dd > 0 ? dot(sub(p, s0), d) / dd : 0.0;
    t = t < 0 ? 0 : (t > 1 ? 1 : t);
    const D3 r = sub(p, add(s0, mul(d, t)));
    return std::sqrt(dot(r, r));
}

// float64 distance from p to the triangle (a, b, c): the projection when it falls inside, else the nearest edge
static double refDist(D3 p, D3 a, D3 b, D3 c)
{
    double best = std::fmin(segDist(p, a, b), std::fmin(segDist(p, a, c), segDist(p, b, c)));
    const D3 n = cross(sub(b, a), sub(c, a));
    const double nn = dot(n, n);
    if (nn > 0)
    {
        const D3 q = sub(p, mul(n, dot(sub(p, a), n) / nn));
        if (dot(cross(sub(b, a), sub(q, a)), n) >= 0 && dot(cross(sub(c, b), sub(q, b)), n) >= 0 && dot(cross(sub(a, c), sub(q, c)), n) >= 0)
        {
            const D3 r = sub(p, q);
            best = std::fmin(best, std::sqrt(dot(r, r)));
        }
    }
    return best;
}

int main(int argc, char **argv)
{
    const unsigned long long seed = argc > 1 ? strtoull(argv[1], nullptr, 10) : 1;
    const long long want = argc > 2 ? atoll(argv[2]) : 200000;
    std::mt19937_64 rng(seed);
    std::uniform_real_distribution<double> U(0.0, 1.0);
    auto u = [&](double lo, double hi) { return lo + (hi - lo) * U(rng); };
    auto logu = [&](double lo, double hi) { return std::exp(u(std::log(lo), std::log(hi))); };
    long long checked = 0, notBox = 0, notLemma = 0, notFinite = 0, notClose = 0, degenerate = 0, onVertex = 0, onEdge = 0,
              inPlane = 0, kinds[8] = {0};
    double worst = 0.0;
    for (long long it = 0; it < want; it++)
    {
        const int kind = (int)(it % 8);
        kinds[kind]++;
        // centre and size: offsets up to 1e6, extents from 1e-6 to 1e2
        const double off = kind == 6 ? logu(1e3, 1e6) : logu(1e-3, 1e4);
        const double ext = kind == 6 ? logu(1e-6, 1e-1) : logu(1e-4, 1e2);
        float v[9];
        D3 cen = {u(-off, off), u(-off, off), u(-off, off)};
        auto rnd = [&]() { return D3{u(-1, 1), u(-1, 1), u(-1, 1)}; };
        D3 P[3] = {rnd(), rnd(), rnd()};
        switch (kind)
        {
        case 1: // sliver: c close to the line ab
            P[2] = add(mul(add(P[0], P[1]), 0.5 + u(-0.4, 0.4) * 2), mul(rnd(), logu(1e-9, 1e-2)));
            break;
        case 2: // zero area: c exactly a or b, or all three equal
            if (it % 3 == 0) P[2] = P[0]; else if (it % 3 == 1) P[1] = P[2]; else P[1] = P[2] = P[0];
            break;
        case 3: // collinear: c on the line ab (beyond, between)
            P[2] = add(P[0], mul(sub(P[1], P[0]), u(-2, 3)));
            break;
        case 4: // axis-flat: one coordinate equal for all three vertices
        {
            const int ax = (int)(it / 8 % 3);
            const double s = u(-1, 1);
            for (D3 &q : P) (ax == 0 ? q.x : ax == 1 ? q.y : q.z) = s;
            break;
        }
        case 5: // repeated vertex after the float rounding: b within an ulp of a
            P[1] = add(P[0], mul(rnd(), 1e-9));
            break;
        default:
            break;
        }
        for (int k = 0; k < 3; k++)
        {
            v[3 * k] = (float)(cen.x + P[k].x * ext);
            v[3 * k + 1] = (float)(cen.y + P[k].y * ext);
            v[3 * k + 2] = (float)(cen.z + P[k].z * ext);
        }
        // the packed record, as k_pack_triangles writes it
        float t[12];
        for (int i = 0; i < 3; i++) { t[i] = v[i]; t[3 + i] = v[i] - v[3 + i]; t[6 + i] = v[i] - v[6 + i]; t[9 + i] = 0.0f; }
        const D3 A = {v[0], v[1], v[2]}, B = {v[3], v[4], v[5]}, Cv = {v[6], v[7], v[8]};
        // the vertices the function works on: b' = fl(a - e1), c' = fl(a - e2)
        const D3 Br = {(float)(t[0] - t[3]), (float)(t[1] - t[4]), (float)(t[2] - t[5])};
        const D3 Cr = {(float)(t[0] - t[6]), (float)(t[1] - t[7]), (float)(t[2] - t[8])};
        // the point: near, far, on a vertex, on an edge, exactly in the plane
        float p[3];
        const int pk = (int)(it / 8 % 6);
        const double w0 = U(rng), w1 = U(rng) * (1 - w0);
        const D3 in = add(add(mul(A, 1 - w0 - w1), mul(B, w0)), mul(Cv, w1));
        D3 pd;
        if (pk == 0) pd = add(in, mul(rnd(), ext * logu(1e-4, 1.0)));
        else if (pk == 1) pd = add(in, mul(rnd(), ext * logu(1.0, 1e3)));
        else if (pk == 2) { pd = (it & 1) ? B : Cv; onVertex++; }
        else if (pk == 3) { pd = add(A, mul(sub(B, A), U(rng))); onEdge++; }
        else if (pk == 4) { pd = in; inPlane++; }
        else pd = add(in, mul(cross(sub(B, A), sub(Cv, A)), u(-1, 1) / std::fmax(ext, 1e-30)));
        p[0] = (float)pd.x; p[1] = (float)pd.y; p[2] = (float)pd.z;
        float q[3];
        const float d2 = rtb_closest::closestPoint(p, t, q);
        float lo[3], hi[3];
        rtb_bvh::leafBox(v, lo, hi);
        checked++;
        bool bad = false;
        if (!(std::isfinite(q[0]) && std::isfinite(q[1]) && std::isfinite(q[2]) && std::isfinite(d2))) { notFinite++; bad = true; }
        for (int i = 0; i < 3; i++)
            if (!(q[i] >= lo[i] && q[i] <= hi[i])) { notBox++; bad = true; break; }
        if (!(rtb_closest::boxDist2(p, lo, hi) <= d2)) { notLemma++; bad = true; }
        const D3 pp = {p[0], p[1], p[2]};
        const double ref = refDist(pp, A, Br, Cr);
        double extent = 0;
        for (int i = 0; i < 3; i++) extent = std::fmax(extent, (double)hi[i] - (double)lo[i]);
        // the float coordinates of q and p carry a rounding of their magnitude, whatever the triangle's size
        const double mag = std::fmax(std::fmax(std::fabs(A.x), std::fabs(A.y)), std::fmax(std::fabs(A.z), std::fabs((double)p[0])));
        const double mag2 = std::fmax(mag, std::fmax(std::fabs((double)p[1]), std::fabs((double)p[2])));
        const double err = std::fmax(std::fabs(std::sqrt((double)d2) - ref) - ULPS * std::ldexp(mag2, -24), 0.0);
        const double rel = err / (std::sqrt(dot(sub(pp, A), sub(pp, A))) + extent);
        if (rel > worst) worst = rel;
        if (!(rel <= TOL)) { notClose++; bad = true; }
        {
            const float ab[3] = {-t[3], -t[4], -t[5]}, ac[3] = {-t[6], -t[7], -t[8]};
            const float n[3] = {ab[1] * ac[2] - ab[2] * ac[1], ab[2] * ac[0] - ab[0] * ac[2], ab[0] * ac[1] - ab[1] * ac[0]};
            if (n[0] == 0 && n[1] == 0 && n[2] == 0) degenerate++;
        }
        if (bad && notBox + notLemma + notFinite + notClose <= 10)
            printf("violation kind %d point %d: v %.9g %.9g %.9g / %.9g %.9g %.9g / %.9g %.9g %.9g p %.9g %.9g %.9g q %.9g %.9g %.9g "
                   "d %.9g ref %.9g\n", kind, pk, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8], p[0], p[1], p[2], q[0], q[1],
                   q[2], std::sqrt((double)d2), ref);
    }
    printf("random %lld sliver %lld zero_area %lld collinear %lld axis_flat %lld repeated %lld offset %lld\n", kinds[0] + kinds[7],
           kinds[1], kinds[2], kinds[3], kinds[4], kinds[5], kinds[6]);
    printf("worst_relative_error %.3g tolerance %.3g\n", worst, TOL);
    printf("checked %lld on_vertex %lld on_edge %lld in_plane %lld zero_cross %lld not_in_box %lld lemma %lld not_finite %lld "
           "not_close %lld violations %lld\n", checked, onVertex, onEdge, inPlane, degenerate, notBox, notLemma, notFinite, notClose,
           notBox + notLemma + notFinite + notClose);
    return (notBox + notLemma + notFinite + notClose) ? 1 : 0;
}
