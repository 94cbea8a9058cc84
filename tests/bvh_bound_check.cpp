// CPU check of the mesh node test (csrc/rtb_bvh.h), compiled by tests/test_mesh.py with g++ -O2 -ffp-contract=off.
//
// Draws random (ray, triangle) pairs -- triangles from 1e-3 to 1e2 in size and up to 1e4 from the origin, rays aimed at
// points inside and just outside the triangle (the reference's -1e-4 slack), from 1e-2 to 1e4 triangle sizes away, in
// random, nearly grazing, axis-parallel (zero components) and denormal-component directions -- and keeps the pairs the
// reference's test (Triangle.cpp:38-121, restated below in its operation order) ACCEPTS outside the grazing band.  For each
// such pair the node test must visit the triangle's leaf box and enclosing boxes with best = the accepted t.
// usage: bvh_bound_check <seed> <pairs>; prints the counts, exit status 1 on a violation.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <random>

#include "../win32-ray-tracing-demo_b200/csrc/rtb_bvh.h"

static float det3(float a11, float a12, float a13, float a21, float a22, float a23, float a31, float a32, float a33)
{
    return a11 * a22 * a33 + a12 * a23 * a31 + a13 * a21 * a32 - a13 * a22 * a31 - a11 * a23 * a32 - a12 * a21 * a33;
}

// reference Triangle::intersect; v = a, b, c; detM out for the band
static bool refIntersect(const float *v, const float *o, const float *d, float &tOut, float &detOut)
{
    const float m11 = v[0] - v[3], m21 = v[1] - v[4], m31 = v[2] - v[5];
    const float m12 = v[0] - v[6], m22 = v[1] - v[7], m32 = v[2] - v[8];
    const float m13 = d[0], m23 = d[1], m33 = d[2];
    const float b1 = v[0] - o[0], b2 = v[1] - o[1], b3 = v[2] - o[2];
    const float detM = det3(m11, m12, m13, m21, m22, m23, m31, m32, m33);
    detOut = detM;
    if (std::fabs(detM) < 1e-10f) return false;
    const float t = det3(m11, m12, b1, m21, m22, b2, m31, m32, b3) / detM;
    if (t < 0.0005f) return false;
    const float beta = det3(b1, m12, m13, b2, m22, m23, b3, m32, m33) / detM;
    if (beta < -0.0001f || beta > 1.0001f) return false;
    const float gamma = det3(m11, b1, m13, m21, b2, m23, m31, b3, m33) / detM;
    if (gamma < -0.0001f || gamma > 1.0001f || 1 - beta - gamma < -0.0001f || 1 - beta - gamma > 1.0001f) return false;
    tOut = t;
    return true;
}

// grazing band of rtb_bvh.h: |detM_r| <= C kappa_g, kappa_g = 2^-19 dmx (A1 + E^2), in double
static bool inBand(const float *v, const float *d, float detM)
{
    double e1[3], e2[3];
    for (int i = 0; i < 3; i++) { e1[i] = std::fabs((double)(v[i] - v[3 + i])); e2[i] = std::fabs((double)(v[i] - v[6 + i])); }
    const double a1 = e1[0] * (e2[1] + e2[2]) + e1[1] * (e2[0] + e2[2]) + e1[2] * (e2[0] + e2[1]);
    const double e = std::fmax(e1[0] + e1[1] + e1[2], e2[0] + e2[1] + e2[2]);
    const double dmx = std::fmax(std::fabs((double)d[0]), std::fmax(std::fabs((double)d[1]), std::fabs((double)d[2])));
    return std::fabs((double)detM) <= (double)RTB_BVH_C * std::ldexp(1.0, -19) * dmx * (a1 + e * e);
}

int main(int argc, char **argv)
{
    const unsigned long long seed = argc > 1 ? strtoull(argv[1], nullptr, 10) : 1;
    const long long want = argc > 2 ? atoll(argv[2]) : 200000;
    std::mt19937_64 rng(seed);
    std::uniform_real_distribution<double> U(0.0, 1.0);
    auto u = [&](double lo, double hi) { return lo + (hi - lo) * U(rng); };
    long long drawn = 0, accepted = 0, band = 0, checked = 0, zeroDir = 0, denormDir = 0, grazing = 0, outsideTri = 0, bad = 0;
    while (checked < want && drawn < want * 200)
    {
        drawn++;
        const double s = std::pow(10.0, u(-3, 2));
        double O[3];
        const double off = U(rng) < 0.3 ? 0.0 : std::pow(10.0, u(0, 4));
        for (int i = 0; i < 3; i++) O[i] = off * u(-1, 1);
        double V[9];
        for (int i = 0; i < 9; i++) V[i] = O[i % 3] + s * u(-1, 1);
        float v[9];
        for (int i = 0; i < 9; i++) v[i] = (float)V[i];
        // aim point: barycentric weights in [-2e-4, 1 + 2e-4]
        double wb = u(-2e-4, 1.0002), wc = u(-2e-4, 1.0002 - wb);
        if (U(rng) < 0.3) wb = -1e-4 * u(0.99, 1.0); // on the edge of the reference's slack
        if (U(rng) < 0.1) wc = -1e-4 * u(0.99, 1.0);
        const double wa = 1 - wb - wc;
        double P[3], n[3], e1[3], e2[3];
        for (int i = 0; i < 3; i++)
        {
            P[i] = wa * V[i] + wb * V[3 + i] + wc * V[6 + i];
            e1[i] = V[3 + i] - V[i];
            e2[i] = V[6 + i] - V[i];
        }
        n[0] = e1[1] * e2[2] - e1[2] * e2[1]; n[1] = e1[2] * e2[0] - e1[0] * e2[2]; n[2] = e1[0] * e2[1] - e1[1] * e2[0];
        const double nn = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
        if (!(nn > 0)) continue;
        for (double &x : n) x /= nn;
        double D[3];
        const double kind = U(rng);
        int special = 0;
        if (kind < 0.25)
        { // nearly grazing: in-plane direction tilted by 10^-6 .. 1
            double t[3] = {u(-1, 1), u(-1, 1), u(-1, 1)};
            const double dn = t[0] * n[0] + t[1] * n[1] + t[2] * n[2];
            const double tilt = std::pow(10.0, u(-6, 0)) * (U(rng) < 0.5 ? -1 : 1);
            for (int i = 0; i < 3; i++) D[i] = t[i] - dn * n[i] + tilt * n[i];
            special = 1;
        }
        else if (kind < 0.40)
        { // one or two zero components
            for (int i = 0; i < 3; i++) D[i] = u(-1, 1);
            D[rng() % 3] = 0.0;
            if (U(rng) < 0.5) D[rng() % 3] = 0.0;
            special = 2;
        }
        else
            for (int i = 0; i < 3; i++) D[i] = u(-1, 1);
        const double dl = std::sqrt(D[0] * D[0] + D[1] * D[1] + D[2] * D[2]);
        if (!(dl > 0)) continue;
        float d[3];
        for (int i = 0; i < 3; i++) d[i] = (float)(D[i] / dl);
        if (kind >= 0.40 && kind < 0.50)
        { // a denormal component
            d[rng() % 3] = (float)(u(-1, 1) * 1e-39);
            special = 3;
        }
        const double dist = s * std::pow(10.0, u(-2, 4));
        float o[3];
        for (int i = 0; i < 3; i++) o[i] = (float)(P[i] - (double)d[i] * dist);
        float t, detM;
        if (!refIntersect(v, o, d, t, detM)) continue;
        accepted++;
        if (inBand(v, d, detM)) { band++; continue; }
        checked++;
        zeroDir += special == 2;
        denormDir += special == 3;
        grazing += special == 1;
        if (wb < 0 || wc < 0 || wa < 0) outsideTri++;
        float lo[3], hi[3];
        rtb_bvh::leafBox(v, lo, hi);
        const rtb_bvh::Ray R = rtb_bvh::makeRay(o[0], o[1], o[2], d[0], d[1], d[2]);
        bool ok = rtb_bvh::nodeHit(R, lo, hi, t);
        // an enclosing node: the leaf box joined with a random box nearby
        float elo[3], ehi[3];
        for (int i = 0; i < 3; i++)
        {
            const float a = (float)(O[i] + s * u(-5, 5)), b = (float)(O[i] + s * u(-5, 5));
            elo[i] = std::fmin(lo[i], std::fmin(a, b));
            ehi[i] = std::fmax(hi[i], std::fmax(a, b));
        }
        ok = ok && rtb_bvh::nodeHit(R, elo, ehi, t);
        if (!ok)
        {
            if (bad < 10)
                printf("VIOLATION tri %.9g %.9g %.9g  %.9g %.9g %.9g  %.9g %.9g %.9g  o %.9g %.9g %.9g  d %.9g %.9g %.9g  t %.9g\n", v[0], v[1],
                       v[2], v[3], v[4], v[5], v[6], v[7], v[8], o[0], o[1], o[2], d[0], d[1], d[2], t);
            bad++;
        }
    }
    printf("drawn %lld accepted %lld band %lld checked %lld grazing %lld zero_dir %lld denormal_dir %lld outside_triangle %lld "
           "violations %lld\n", drawn, accepted, band, checked, grazing, zeroDir, denormDir, outsideTri, bad);
    return (bad == 0 && checked >= want) ? 0 : 1;
}
