// CPU check of the winding-number math (csrc/rtb_winding.h), compiled by tests/test_winding.py with
// g++ -O2 -std=c++17 -ffp-contract=off.
//
//   * atan2 against double atan2 within RTB_ATAN2_REL relative (plus 2^-126 absolute where the float result is below the
//     normal range), over both axes, signed zeros, infinities, a dense sweep of y / x in [0, 1] and random pairs whose
//     ratios span 2^-280 .. 2^280, in all four quadrants;
//   * solidAngle against a float64 evaluation on the same float vertices (a, b' = fl(a + ab), c' = fl(a + ac)) within
//     RTB_SOLID_ABS + RTB_SOLID_COND L / D modulo 4 pi (rtb_winding.h), on random and adversarial triangles -- slivers,
//     zero-area, collinear, repeated vertices, coordinates offset up to 1e4 -- with points near and far, on vertices, on
//     edges and in the triangle's plane; and that every output is finite;
//   * closed soups -- a tetrahedron, a cube and a tessellated sphere, at several offsets and scales -- summed as the kernel
//     sums (w += fl(Omega * fl(1 / 4 pi)) in order): 1 inside and 0 outside within the sum of the per-triangle bounds / 4 pi
//     plus the summation bound m 2^-24 sum |Omega| / 4 pi.
// usage: winding_check <seed> <pairs>; prints the counts and the worst errors, exit status 1 on a violation.
#include <array>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>

#include "../win32-ray-tracing-demo_b200/csrc/rtb_winding.h"

using rtb_winding::solidAngle;

struct D3 { double x, y, z; };
static D3 sub(D3 a, D3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
static double dot(D3 a, D3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static D3 cross(D3 a, D3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
static double len(D3 a) { return std::sqrt(dot(a, a)); }

static long violations = 0;
static double worstAtan = 0, worstSolid = 0, worstSolidAbs = 0, worstSum = 0;

static void checkAtan(float y, float x)
{
    const float r = rtb_winding::atan2(y, x);
    const double ref = std::atan2((double)y, (double)x);
    if (std::isnan(ref)) { if (!std::isnan(r)) { violations++; printf("atan2(%a, %a) = %a, want NaN\n", y, x, r); } return; }
    const double err = std::fabs((double)r - ref);
    const double rel = ref != 0 ? err / std::fabs(ref) : (err == 0 ? 0 : INFINITY);
    if (std::fabs(ref) >= 0x1p-126) worstAtan = std::fmax(worstAtan, rel);
    if (!(err <= RTB_ATAN2_REL * std::fabs(ref) + 0x1p-126) || std::signbit(r) != std::signbit(ref))
    {
        violations++;
        if (violations < 20) printf("atan2(%a, %a) = %.9g, want %.17g\n", y, x, r, ref);
    }
}

// packed record {a, e1 = fl(a - b), e2 = fl(a - c), n} as k_pack_triangles writes it
static void pack(const float v[9], float t[12])
{
    for (int i = 0; i < 3; i++) { t[i] = v[i]; t[3 + i] = v[i] - v[3 + i]; t[6 + i] = v[i] - v[6 + i]; t[9 + i] = 0.0f; }
}

// float64 solid angle on the float vertices the header uses; L = |A||B||C|, D = hypot(det, den)
static double refSolid(const float p[3], const float t[12], double &L, double &D)
{
    const D3 P = {p[0], p[1], p[2]};
    const D3 a = {t[0], t[1], t[2]};
    const D3 b = {(float)(t[0] + -t[3]), (float)(t[1] + -t[4]), (float)(t[2] + -t[5])};
    const D3 c = {(float)(t[0] + -t[6]), (float)(t[1] + -t[7]), (float)(t[2] + -t[8])};
    const D3 A = sub(a, P), B = sub(b, P), C = sub(c, P);
    const double la = len(A), lb = len(B), lc = len(C);
    const double det = dot(A, cross(B, C));
    const double den = la * lb * lc + dot(A, B) * lc + dot(A, C) * lb + dot(B, C) * la;
    L = la * lb * lc;
    D = std::hypot(det, den);
    return 2 * std::atan2(det, den);
}

static double solidBound(double L, double D) { return RTB_SOLID_ABS + RTB_SOLID_COND * (D > 0 ? L / D : INFINITY); }

static void checkSolid(const float p[3], const float t[12], long &checked)
{
    const float s = solidAngle(p, t);
    double L, D;
    const double ref = refSolid(p, t, L, D);
    checked++;
    if (!std::isfinite(s)) { violations++; printf("solidAngle not finite: %a\n", s); return; }
    if (!(D > 0)) return; // p on a vertex: any value (the header returns 0 when its det and den are 0)
    const double err = std::fabs(std::remainder((double)s - ref, 4 * M_PI));
    const double bound = solidBound(L, D);
    worstSolid = std::fmax(worstSolid, err / bound);
    if (L / D < 4) worstSolidAbs = std::fmax(worstSolidAbs, err);
    if (!(err <= bound))
    {
        violations++;
        if (violations < 20) printf("solidAngle %.9g, want %.17g (L/D %.3g, bound %.3g)\n", s, ref, L / D, bound);
    }
}

// ---- closed soups -----------------------------------------------------------------------------
using Soup = std::vector<std::array<float, 9>>;

static Soup tetrahedron()
{
    const float v[4][3] = {{1, 1, 1}, {1, -1, -1}, {-1, 1, -1}, {-1, -1, 1}};
    const int f[4][3] = {{0, 1, 2}, {0, 3, 1}, {0, 2, 3}, {1, 3, 2}}; // outward: (b - a) x (c - a) away from the centre
    Soup s;
    for (auto &t : f) s.push_back({v[t[0]][0], v[t[0]][1], v[t[0]][2], v[t[1]][0], v[t[1]][1], v[t[1]][2], v[t[2]][0], v[t[2]][1], v[t[2]][2]});
    return s;
}

static Soup cube()
{
    Soup s;
    for (int ax = 0; ax < 3; ax++)
        for (int sg = -1; sg <= 1; sg += 2)
        { // face at coordinate ax = sg; u, v the other axes, ordered so that u x v = sg e_ax
            const int u = (ax + 1) % 3, w = (ax + 2) % 3;
            float q[4][3];
            const float uu[4] = {-1, 1, 1, -1}, vv[4] = {-1, -1, 1, 1};
            for (int k = 0; k < 4; k++) { q[k][ax] = (float)sg; q[k][u] = uu[k]; q[k][w] = vv[k] * (float)sg; }
            auto tri = [&](int a, int b, int c) { s.push_back({q[a][0], q[a][1], q[a][2], q[b][0], q[b][1], q[b][2], q[c][0], q[c][1], q[c][2]}); };
            tri(0, 1, 2);
            tri(0, 2, 3);
        }
    return s;
}

static Soup sphere(int nu, int nv)
{
    auto pt = [&](int i, int j, float o[3]) {
        const double u = 2 * M_PI * i / nu, v = M_PI * j / nv;
        o[0] = (float)(std::sin(v) * std::cos(u)); o[1] = (float)(std::sin(v) * std::sin(u)); o[2] = (float)std::cos(v);
    };
    Soup s;
    for (int i = 0; i < nu; i++)
        for (int j = 0; j < nv; j++)
        {
            float a[3], b[3], c[3], d[3];
            pt(i, j, a); pt(i, j + 1, b); pt(i + 1, j + 1, c); pt(i + 1, j, d);
            if (j > 0) s.push_back({a[0], a[1], a[2], b[0], b[1], b[2], d[0], d[1], d[2]});          // outward: a b d
            if (j < nv - 1) s.push_back({b[0], b[1], b[2], c[0], c[1], c[2], d[0], d[1], d[2]});
        }
    return s;
}

static void checkSoup(const char *name, const Soup &soup0, double inR, double outR, std::mt19937_64 &g, long &sums)
{
    std::uniform_real_distribution<double> U(-1, 1);
    const double offsets[3] = {0, 37.5, 1000};
    const double scales[3] = {1, 0.01, 300};
    for (double off : offsets)
        for (double sc : scales)
        {
            std::vector<float> packed;
            for (auto &v : soup0)
            {
                float w[9], t[12];
                for (int i = 0; i < 9; i++) w[i] = (float)(v[i] * sc + off);
                pack(w, t);
                packed.insert(packed.end(), t, t + 12);
            }
            const size_t m = soup0.size();
            for (int k = 0; k < 400; k++)
            {
                D3 d;
                do d = {U(g), U(g), U(g)}; while (dot(d, d) > 1 || dot(d, d) < 1e-6);
                const bool in = k & 1;
                const double rad = in ? inR * (0.05 + 0.95 * U(g) * U(g)) : outR * (1 + 4 * std::fabs(U(g)));
                const double n = len(d);
                const float p[3] = {(float)(d.x / n * rad * sc + off), (float)(d.y / n * rad * sc + off), (float)(d.z / n * rad * sc + off)};
                float w = 0.0f;
                double bound = 0, absSum = 0;
                for (size_t j = 0; j < m; j++)
                {
                    const float om = solidAngle(p, &packed[12 * j]);
                    w += om * RTB_WINDING_INV4PI;
                    double L, D;
                    refSolid(p, &packed[12 * j], L, D);
                    bound += solidBound(L, D) / (4 * M_PI);
                    absSum += std::fabs(om) / (4 * M_PI);
                }
                bound += (double)m * 0x1p-24 * absSum;
                const double err = std::fabs((double)w - (in ? 1.0 : 0.0));
                worstSum = std::fmax(worstSum, err);
                sums++;
                if (!(err <= bound))
                {
                    violations++;
                    if (violations < 20) printf("%s: w %.9g at (%g %g %g), inside %d, bound %.3g\n", name, w, p[0], p[1], p[2], in, bound);
                }
            }
        }
}

int main(int argc, char **argv)
{
    const unsigned long long seed = argc > 1 ? strtoull(argv[1], nullptr, 10) : 1;
    const long pairs = argc > 2 ? atol(argv[2]) : 100000;
    std::mt19937_64 g(seed);
    std::uniform_real_distribution<double> U(0, 1);

    // ---- atan2 ----
    long atans = 0;
    const float specials[] = {0.0f, -0.0f, 1.0f, -1.0f, 0x1p-149f, -0x1p-149f, 0x1p-126f, 3.4028235e38f, -3.4028235e38f, INFINITY, -INFINITY, NAN};
    for (float y : specials)
        for (float x : specials) { checkAtan(y, x); atans++; }
    for (long k = 0; k <= (1 << 24); k++)
    { // y / x = k 2^-24 over [0, 1], and the mirrored octants
        const float y = (float)k * 0x1p-24f;
        checkAtan(y, 1.0f); checkAtan(1.0f, y); checkAtan(-y, -1.0f); checkAtan(y, -1.0f);
        atans += 4;
    }
    for (long k = 0; k < 4 * pairs; k++)
    {
        const float y = (float)((U(g) + 0.5) * std::ldexp(1.0, (int)(U(g) * 280) - 140)) * (U(g) < 0.5 ? -1.0f : 1.0f);
        const float x = (float)((U(g) + 0.5) * std::ldexp(1.0, (int)(U(g) * 280) - 140)) * (U(g) < 0.5 ? -1.0f : 1.0f);
        checkAtan(y, x);
        checkAtan(y, U(g) < 0.5 ? 0.0f : -0.0f);
        checkAtan(U(g) < 0.5 ? 0.0f : -0.0f, x);
        atans += 3;
    }

    // ---- solid angles ----
    long checked = 0, onVertex = 0, onEdge = 0, inPlane = 0, degenerate = 0;
    for (long k = 0; k < pairs; k++)
    {
        const double off = U(g) < 0.3 ? std::pow(10.0, U(g) * 4) * (U(g) < 0.5 ? -1 : 1) : 0.0;
        const double ext = std::pow(10.0, -3 + U(g) * 5);
        float v[9];
        for (int i = 0; i < 9; i++) v[i] = (float)(off + (U(g) - 0.5) * ext);
        const int kind = (int)(U(g) * 8);
        if (kind == 1) { for (int i = 0; i < 3; i++) v[3 + i] = v[i]; degenerate++; }                         // repeated vertex
        else if (kind == 2) { for (int i = 0; i < 3; i++) v[6 + i] = (float)(v[i] + (v[3 + i] - v[i]) * (U(g) * 3 - 1)); degenerate++; } // collinear
        else if (kind == 3) { for (int i = 0; i < 3; i++) v[6 + i] = (float)(v[i] + (v[3 + i] - v[i]) * 0.5 + (U(g) - 0.5) * ext * 1e-5); degenerate++; } // sliver
        else if (kind == 4) { for (int i = 0; i < 9; i++) v[i] = (float)off; degenerate++; }                   // a point
        float t[12];
        pack(v, t);
        const float a[3] = {t[0], t[1], t[2]};
        const float b[3] = {t[0] + -t[3], t[1] + -t[4], t[2] + -t[5]}, c[3] = {t[0] + -t[6], t[1] + -t[7], t[2] + -t[8]};
        float p[3];
        const int where = (int)(U(g) * 6);
        const double near = ext * std::pow(10.0, -6 + U(g) * 7);
        if (where == 0) { const float *s = U(g) < 0.34 ? a : (U(g) < 0.5 ? b : c); for (int i = 0; i < 3; i++) p[i] = s[i]; onVertex++; }
        else if (where == 1)
        { // on an edge (rounded to float)
            const double s = U(g);
            for (int i = 0; i < 3; i++) p[i] = (float)(a[i] + (b[i] - (double)a[i]) * s);
            onEdge++;
        }
        else if (where == 2)
        { // in the plane: a + s ab + u ac, inside or outside the triangle
            const double s = U(g) * 1.4 - 0.2, u = U(g) * 1.4 - 0.2;
            for (int i = 0; i < 3; i++) p[i] = (float)(a[i] + (b[i] - (double)a[i]) * s + (c[i] - (double)a[i]) * u);
            inPlane++;
        }
        else if (where == 3)
        { // near the surface, both sides
            const double s = U(g), u = U(g) * (1 - s);
            const D3 n = cross(sub({b[0], b[1], b[2]}, {a[0], a[1], a[2]}), sub({c[0], c[1], c[2]}, {a[0], a[1], a[2]}));
            const double nl = len(n) > 0 ? len(n) : 1;
            const double h = (U(g) < 0.5 ? -near : near) / nl;
            p[0] = (float)(a[0] + (b[0] - (double)a[0]) * s + (c[0] - (double)a[0]) * u + n.x * h);
            p[1] = (float)(a[1] + (b[1] - (double)a[1]) * s + (c[1] - (double)a[1]) * u + n.y * h);
            p[2] = (float)(a[2] + (b[2] - (double)a[2]) * s + (c[2] - (double)a[2]) * u + n.z * h);
        }
        else
        { // anywhere from near to far
            const double r = ext * std::pow(10.0, -2 + U(g) * 5);
            for (int i = 0; i < 3; i++) p[i] = (float)(a[i] + (U(g) - 0.5) * r);
        }
        checkSolid(p, t, checked);
    }

    // ---- closed soups ----
    long sums = 0;
    checkSoup("tetrahedron", tetrahedron(), 0.5, 3.0, g, sums);
    checkSoup("cube", cube(), 0.99, 1.75, g, sums);
    checkSoup("sphere", sphere(48, 24), 0.99 * std::cos(M_PI / 24), 1.01, g, sums);

    printf("worst atan2 rel %.3g (bound %.3g); worst solidAngle err / bound %.3g, abs err where L/D < 4: %.3g; worst |w - w_exact| %.3g\n",
           worstAtan, (double)RTB_ATAN2_REL, worstSolid, worstSolidAbs, worstSum);
    printf("atan2 %ld checked %ld on_vertex %ld on_edge %ld in_plane %ld degenerate %ld sums %ld violations %ld\n", atans, checked,
           onVertex, onEdge, inPlane, degenerate, sums, violations);
    return violations ? 1 : 0;
}
