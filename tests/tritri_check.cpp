// CPU check of the triangle-query overlap test (csrc/rtb_tritri.h), compiled by tests/test_triangle_query.py with
// g++ -O2 -std=c++17 -ffp-contract=off.
//
// Draws seeded pairs of triangles of ten kinds: random; a shared vertex; a shared edge; a vertex on the other's face and two
// edges crossing at one point (dyadic coordinates, so the contact is exact in float); coplanar pairs on an integer grid
// (overlapping, touching or disjoint); a touching pair with one coordinate moved by one ulp; coordinates offset up to 1e6 with
// extents down to 1e-6; denormal coordinates; and degenerate triangles (collinear, repeated vertices, non-finite).  For each
// pair it checks:
//   * a degenerate triangle intersects nothing;
//   * boxes the box test separates hold no intersecting pair (the pruning lemma);
//   * the answer does not change when the two triangles are swapped, or the vertices of either are rotated or reversed;
//   * the constructed contacts (shared vertex or edge, vertex on a face, crossing edges) are reported.
// The exact answer is checked independently by the Fraction oracle of tests/test_triangle_query.py on the pairs dumped here.
// usage: tritri_check <seed> <pairs> [dump file]; the dump holds per pair p[9], q[9] (float32), the answer, whether an exact
// fallback ran and the kind (uint8 each).  Prints the counts; exit status 1 on a violation.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>

static long g_exact[4];
#define RTB_TRITRI_COUNT(k) (++g_exact[k])
#include "../win32-ray-tracing-demo_b200/csrc/rtb_tritri.h"

enum { RANDOM, SHARED_VERTEX, SHARED_EDGE, ON_FACE, CROSSING, COPLANAR, ONE_ULP, OFFSET, DENORMAL, DEGENERATE, KINDS };

static std::mt19937_64 rng;
static double uni(double lo, double hi) { return std::uniform_real_distribution<double>(lo, hi)(rng); }
static int irand(int lo, int hi) { return std::uniform_int_distribution<int>(lo, hi)(rng); }

static void randomTri(float *t, double lo, double hi)
{
    for (int i = 0; i < 9; i++) t[i] = (float)uni(lo, hi);
}
static void gridTri(float *t, int r)
{
    for (int i = 0; i < 9; i++) t[i] = (float)irand(-r, r);
}

// a pair that touches by construction (kinds SHARED_VERTEX .. CROSSING), on an integer grid scaled by 4 so that the midpoints
// and face points below are exact
static void contactPair(int kind, float *p, float *q)
{
    gridTri(p, 8);
    gridTri(q, 8);
    for (int i = 0; i < 9; i++) { p[i] *= 4; q[i] *= 4; }
    const int v = irand(0, 2), w = (v + 1) % 3;
    if (kind == SHARED_VERTEX) std::memcpy(q + 3 * irand(0, 2), p + 3 * v, 12);
    else if (kind == SHARED_EDGE)
    {
        const bool flip = irand(0, 1);
        std::memcpy(q + (flip ? 3 : 0), p + 3 * v, 12);
        std::memcpy(q + (flip ? 0 : 3), p + 3 * w, 12);
    }
    else if (kind == ON_FACE) // q's first vertex at (p0 + p1 + 2 p2) / 4, or on an edge, or the centre of an edge
    {
        const int wa = irand(0, 2), wb = irand(0, 4 - wa), wc = 4 - wa - wb;
        for (int i = 0; i < 3; i++) q[i] = (wa * p[i] + wb * p[3 + i] + wc * p[6 + i]) / 4;
    }
    else // two edges crossing at the midpoint of p's edge v -> w: q's edge 0 -> 1 through it
    {
        for (int i = 0; i < 3; i++)
        {
            const float m = (p[3 * v + i] + p[3 * w + i]) / 2, d = (float)irand(-8, 8);
            q[i] = m + d;
            q[3 + i] = m - d;
        }
    }
}

static void coplanarPair(float *p, float *q)
{
    // both in the plane x + y + z = c (or z = c): integer coordinates, so the plane is exact
    const int c = irand(-4, 4), general = irand(0, 1), r = irand(1, 4);
    for (float *t : {p, q})
        for (int j = 0; j < 3; j++)
        {
            const int x = irand(-r, r), y = irand(-r, r);
            t[3 * j] = (float)x; t[3 * j + 1] = (float)y;
            t[3 * j + 2] = (float)(general ? c - x - y : c);
        }
}

static void offsetPair(float *p, float *q)
{
    const double o[3] = {uni(-1e6, 1e6), uni(-1e6, 1e6), uni(-1e6, 1e6)}, ext = std::pow(10.0, uni(-6, 0));
    for (int i = 0; i < 9; i++)
    {
        p[i] = (float)(o[i % 3] + ext * uni(-1, 1));
        q[i] = (float)(o[i % 3] + ext * uni(-1, 1));
    }
    if (irand(0, 1)) std::memcpy(q, p + 3 * irand(0, 2), 12);
}

static void degeneratePair(float *p, float *q)
{
    gridTri(p, 4);
    gridTri(q, 4);
    float *t = irand(0, 1) ? p : q;
    const int how = irand(0, 3);
    if (how == 0) for (int i = 0; i < 3; i++) t[6 + i] = t[i] + 2 * (t[3 + i] - t[i]); // collinear
    else if (how == 1) std::memcpy(t + 3 * irand(1, 2), t, 12);                        // repeated vertex
    else if (how == 2) { std::memcpy(t + 3, t, 12); std::memcpy(t + 6, t, 12); }        // a point
    else t[irand(0, 8)] = irand(0, 1) ? NAN : (irand(0, 1) ? INFINITY : -INFINITY);      // non-finite
    if (irand(0, 1)) std::memcpy(p == t ? q : p, t, 12);                                 // sharing its first vertex
}

static void draw(int kind, float *p, float *q)
{
    switch (kind)
    {
    case RANDOM:
        randomTri(p, -1, 1);
        randomTri(q, -1, 1);
        for (int i = 0; i < 9; i++) q[i] = q[i] * 0.7f + 0.3f;
        break;
    case COPLANAR: coplanarPair(p, q); break;
    case ONE_ULP:
        contactPair(irand(SHARED_VERTEX, CROSSING), p, q);
        {
            float *t = irand(0, 1) ? p : q;
            const int i = irand(0, 8);
            t[i] = std::nextafter(t[i], irand(0, 1) ? INFINITY : -INFINITY);
        }
        break;
    case OFFSET: offsetPair(p, q); break;
    case DENORMAL:
        if (irand(0, 1)) coplanarPair(p, q);
        else contactPair(irand(SHARED_VERTEX, CROSSING), p, q);
        for (int i = 0; i < 9; i++) { p[i] = std::ldexp(p[i], -140); q[i] = std::ldexp(q[i], -140); } // exact: small integers
        break;
    case DEGENERATE: degeneratePair(p, q); break;
    default: contactPair(kind, p, q);
    }
}

// vertex order: rotation r (0..2), reversed or not
static void reorder(const float *t, int r, bool rev, float *out)
{
    for (int j = 0; j < 3; j++)
    {
        const int s = rev ? (r + 3 - j) % 3 : (r + j) % 3;
        std::memcpy(out + 3 * j, t + 3 * s, 12);
    }
}

int main(int argc, char **argv)
{
    if (argc < 3) { std::fprintf(stderr, "usage: tritri_check <seed> <pairs> [dump]\n"); return 2; }
    rng.seed(std::strtoull(argv[1], nullptr, 10));
    const long n = std::atol(argv[2]);
    FILE *dump = argc > 3 ? std::fopen(argv[3], "wb") : nullptr;
    long violations = 0, hits = 0, degenerate = 0, fallbackPairs = 0, exact3 = 0, exact2 = 0, byKind[KINDS] = {}, hitKind[KINDS] = {};
    for (long it = 0; it < n; it++)
    {
        const int kind = (int)(it % KINDS);
        float p[9], q[9];
        draw(kind, p, q);
        const long e0 = g_exact[3] + g_exact[2];
        const bool hit = rtb_tritri::intersect(p, q);
        const bool fell = g_exact[3] + g_exact[2] != e0;
        const bool deg = rtb_tritri::degenerate(p) || rtb_tritri::degenerate(q);
        float plo[3], phi[3], qlo[3], qhi[3];
        rtb_tritri::box(p, plo, phi);
        rtb_tritri::box(q, qlo, qhi);
        bool bad = (deg && hit) || (kind == DEGENERATE && !deg) || (hit && !rtb_tritri::boxesOverlap(plo, phi, qlo, qhi));
        if (!deg && kind >= SHARED_VERTEX && kind <= CROSSING && !hit) bad = true;
        const long x3 = g_exact[3], x2 = g_exact[2]; // the reorderings below do not count as the pair's own evaluations
        for (int r = 0; r < 3 && !bad; r++)
            for (int rev = 0; rev < 2 && !bad; rev++)
            {
                float pp[9], qq[9];
                reorder(p, r, rev, pp);
                reorder(q, (r + rev) % 3, !rev, qq);
                if (rtb_tritri::intersect(pp, qq) != hit || rtb_tritri::intersect(qq, pp) != hit) bad = true;
            }
        g_exact[3] = x3; g_exact[2] = x2;
        if (bad)
        {
            if (violations < 10)
            {
                std::printf("violation kind %d hit %d deg %d p", kind, (int)hit, (int)deg);
                for (float v : p) std::printf(" %.9g", v);
                std::printf(" q");
                for (float v : q) std::printf(" %.9g", v);
                std::printf("\n");
            }
            violations++;
        }
        hits += hit;
        degenerate += deg;
        fallbackPairs += fell;
        byKind[kind]++;
        hitKind[kind] += hit;
        if (dump)
        {
            const unsigned char extra[3] = {(unsigned char)hit, (unsigned char)fell, (unsigned char)kind};
            std::fwrite(p, 4, 9, dump);
            std::fwrite(q, 4, 9, dump);
            std::fwrite(extra, 1, 3, dump);
        }
    }
    exact3 = g_exact[3];
    exact2 = g_exact[2];
    if (dump) std::fclose(dump);
    for (int k = 0; k < KINDS; k++) std::printf("kind %d pairs %ld intersecting %ld\n", k, byKind[k], hitKind[k]);
    std::printf("checked %ld violations %ld intersecting %ld degenerate %ld fallback_pairs %ld exact3 %ld exact2 %ld\n", n, violations,
                hits, degenerate, fallbackPairs, exact3, exact2);
    return violations ? 1 : 0;
}
