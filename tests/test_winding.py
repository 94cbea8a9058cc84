"""rtb_query_winding: generalised winding numbers of points with respect to the scene's TRIANGLES and MESH records, inside /
outside tests and signed distances, on device buffers and ordered on the caller's stream (include/rtb.h, DESIGN 3f).  Oracles:
csrc/rtb_winding.h compiled for the host (its CPU check against float64, and a brute-force sum over it that a TRIANGLES run
must equal bit for bit), the run of the same triangles for a mesh summed exactly (beta = inf), and a float64 numpy brute
force for the approximate walk."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import rtb200
from test_mesh import _ball, _flat, _flat_records, _tris_from_facets
from test_mesh_update import _overlap_layout, twist
from test_point_query import _packed, _torch_points
from test_ray_query import _run_twin

ERR_INVALID = -1
CSRC = os.path.join(rtb200.PKG, "csrc")
INF = float("inf")
OFFSETS = (1e-3, 1e-2, 1e-1, 1.0)  # near-surface offsets, times the mesh's mean edge length
# Stated accuracy of the first-order walk at beta = 2 against float64: max |w - w64| over every band but the vertices (DESIGN
# 3f).  The worst seen on a B200 was 0.036 (the 100 k torus, uniform points) on the closed tori and 0.030 on the open half.
FAST_BOUND = 0.05
OPEN_BOUND = {2.0: 0.05, INF: 1e-3}  # the open half-torus, beta = 2 and beta = inf (exact: float32 rounding only)


# ---- host side (no device) --------------------------------------------------------------------
def test_winding_check_on_the_cpu(tmp_path):
    """csrc/rtb_winding.h for the host: atan2 against double atan2 within its stated bound, solidAngle against float64 within
    its stated bound on random and adversarial triangles, and closed soups summing to 1 inside and 0 outside."""
    exe = str(tmp_path / "winding_check")
    src = os.path.join(rtb200.ROOT, "tests", "winding_check.cpp")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-o", exe, src])
    for seed in (1, 2):
        out = subprocess.run([exe, str(seed), "200000"], capture_output=True, text=True)
        print(out.stdout)
        assert out.returncode == 0, out.stdout
        counts = dict(re.findall(r"(\w+) (\d+)", out.stdout.splitlines()[-1]))
        assert int(counts["violations"]) == 0 and int(counts["checked"]) == 200000 and int(counts["atan2"]) > 60_000_000
        assert int(counts["on_vertex"]) > 10000 and int(counts["on_edge"]) > 10000 and int(counts["in_plane"]) > 10000
        assert int(counts["degenerate"]) > 50000 and int(counts["sums"]) == 10800


def test_header_winding_query_matches_the_bindings():
    text = open(os.path.join(rtb200.ROOT, "include", "rtb.h")).read()
    assert re.search(r"int rtb_scene_mesh_moments\(rtb_ctx \*ctx, rtb_scene \*scene, void \*stream\);", text)
    assert re.search(r"int rtb_query_winding\(rtb_ctx \*ctx, const rtb_scene \*scene, int64_t n, const float \*points, float beta, "
                     r"float \*winding,\s+uint8_t \*inside, void \*stream\);", text)
    assert "rtb_scene_mesh_moments" in rtb200.ABI_SYMBOLS and "rtb_query_winding" in rtb200.ABI_SYMBOLS
    assert "#define RTB_ABI_VERSION 5" in text


# ---- host model: the header compiled into a small library --------------------------------------
_HOST_SRC = r"""
#include "rtb_winding.h"
// brute force over packed records t[m][12] (a, a - b, a - c, n) as one TRIANGLES run, in k order, as the kernel sums;
// abs_sum[i] = sum of |term|, for the summation-order bound
extern "C" void winding_all(const float *t, int m, const float *pts, long n, float *w, double *abs_sum)
{
#pragma omp parallel for schedule(dynamic, 256)
    for (long i = 0; i < n; i++)
    {
        const float *p = pts + 3 * i;
        float s = 0.0f;
        double a = 0.0;
        if (!(p[0] == p[0] && p[1] == p[1] && p[2] == p[2])) s = NAN;
        else
            for (int j = 0; j < m; j++)
            {
                const float term = rtb_winding::solidAngle(p, t + 12 * (long)j) * RTB_WINDING_INV4PI;
                s += term;
                a += term < 0 ? -(double)term : (double)term;
            }
        w[i] = s;
        abs_sum[i] = a;
    }
}
"""


@pytest.fixture(scope="module")
def host_model(tmp_path_factory):
    d = tmp_path_factory.mktemp("winding_host")
    src, so = d / "winding_host.cpp", d / "winding_host.so"
    src.write_text(_HOST_SRC)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC", "-I", CSRC, "-o", str(so),
                           str(src)])
    lib = C.CDLL(str(so))
    vp = C.c_void_p
    lib.winding_all.argtypes = [vp, C.c_int, vp, C.c_long, vp, vp]

    def run(tris, pts):
        packed = _packed(tris)
        pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 3)
        w, a = np.zeros(len(pts), np.float32), np.zeros(len(pts), np.float64)
        lib.winding_all(packed.ctypes.data, len(packed), pts.ctypes.data, len(pts), w.ctypes.data, a.ctypes.data)
        return w, a
    return run


# ---- models and points ------------------------------------------------------------------------
def _torus(n, seed):
    """rtb200.torus_triangles with b and c swapped: its facets then face outwards by the right-hand rule, so w = 1 inside"""
    t = _tris_from_facets(rtb200.torus_triangles(n, seed=seed))
    return np.ascontiguousarray(np.concatenate([t[:, 0:3], t[:, 6:9], t[:, 3:6], -t[:, 9:12]], 1), np.float32)


def _half(tris):
    """an open soup: the facets of the torus on one side of its centre plane x = 0"""
    c = tris[:, :9].reshape(-1, 3, 3).mean(1)
    return np.ascontiguousarray(tris[c[:, 0] > 0], np.float32)


def _edge(tris):
    v = tris[:, :9].reshape(-1, 3, 3).astype(np.float64)
    return float(np.mean(np.linalg.norm(v - np.roll(v, 1, axis=1), axis=2)))


def _points(tris, rng, n_band, n_uniform):
    """(points, band): near the surface at +-OFFSETS x the mean edge length along the facet's right-hand normal (band
    = +-offset, + outside), uniform in the box grown by a tenth (band nan), and on vertices (band 0)"""
    v = tris[:, :9].reshape(-1, 3, 3).astype(np.float64)
    e = _edge(tris)
    pts, band = [], []
    for off in OFFSETS:
        for sgn in (1.0, -1.0):
            k = rng.integers(0, len(v), n_band)
            surf = np.einsum("ni,nij->nj", rng.dirichlet([1, 1, 1], n_band), v[k])
            nrm = np.cross(v[k, 1] - v[k, 0], v[k, 2] - v[k, 0])
            nrm /= np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-30)
            pts.append(surf + nrm * (sgn * off * e))
            band.append(np.full(n_band, sgn * off))
    lo, hi = v.reshape(-1, 3).min(0), v.reshape(-1, 3).max(0)
    pts.append(lo - (hi - lo) * 0.05 + rng.uniform(size=(n_uniform, 3)) * (hi - lo) * 1.1)
    band.append(np.full(n_uniform, np.nan))
    k = rng.integers(0, len(v), n_band)
    pts.append(v[k, rng.integers(0, 3, n_band)])
    band.append(np.zeros(n_band))
    return np.ascontiguousarray(np.concatenate(pts), np.float32), np.concatenate(band)


def _w64(tris, pts, pairs=4_000_000):
    """float64 winding numbers (numpy brute force, van Oosterom--Strackee on the float vertices)"""
    v = tris[:, :9].astype(np.float64)
    out = np.empty(len(pts))
    step = max(1, pairs // len(v))
    for s in range(0, len(pts), step):
        p = np.asarray(pts[s:s + step], np.float64)
        A, B, Cc = ([v[None, :, 3 * k + i] - p[:, i, None] for i in range(3)] for k in range(3))
        la, lb, lc = (np.sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]) for x in (A, B, Cc))
        det = A[0] * (B[1] * Cc[2] - B[2] * Cc[1]) + A[1] * (B[2] * Cc[0] - B[0] * Cc[2]) + A[2] * (B[0] * Cc[1] - B[1] * Cc[0])
        dot = lambda x, y: x[0] * y[0] + x[1] * y[1] + x[2] * y[2]
        den = la * lb * lc + dot(A, B) * lc + dot(A, Cc) * lb + dot(B, Cc) * la
        out[s:s + step] = (2 * np.arctan2(det, den)).sum(1) / (4 * np.pi)
    return out


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


def _bits(x):
    return x.cpu().numpy().view(np.uint32)


@pytest.fixture(scope="module")
def ctx():
    c = rtb200.Context(0)
    yield c
    c.close()


# ---- run == host model, bit for bit; exact mesh == run within the summation bound --------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["torus10k", "ball"])
def test_run_equals_host_and_exact_mesh_equals_run(ctx, host_model, name):
    tris = _torus(10_000, 3) if name == "torus10k" else _ball()
    pts, _ = _points(tris, np.random.default_rng(61), 6144, 65536 - 9 * 6144)
    assert len(pts) == 65536
    run, mesh = ctx.upload(_flat(tris, False)), ctx.upload(_flat(tris, True))
    try:
        pt = _t(pts)
        w_run = run.winding_numbers(pt).cpu().numpy()
        w_host, abs_sum = host_model(tris, pts)
        assert np.array_equal(w_run.view(np.uint32), w_host.view(np.uint32)), \
            f"{name}: the run differs from the host model on {int((w_run.view(np.uint32) != w_host.view(np.uint32)).sum())} points"
        assert np.array_equal(run.contains(pt).cpu().numpy(), w_host > 0.5)
        w_mesh = mesh.winding_numbers(pt, beta=INF).cpu().numpy()
        bound = len(tris) * 2.0 ** -23 * abs_sum
        err = np.abs(w_mesh.astype(np.float64) - w_run)
        print(f"{name}: run == host model on {len(pts)} points; exact mesh - run: worst {err.max():.3g}, "
              f"worst / bound {np.max(err / bound):.3g}")
        assert (err <= bound).all()
    finally:
        run.close()
        mesh.close()


# ---- the fast walk against float64 --------------------------------------------------------------
def _classify(s, tris, pts, band, w, what, bound=FAST_BOUND):
    """contains == the float64 classification at every offset band and for uniform points at least the smallest offset away
    from the surface; max |w - w64| per band printed and below `bound`"""
    w64 = _w64(tris, pts)
    d = s.closest_points(_t(pts))[1].cpu().numpy()
    keep = np.where(np.isnan(band), d >= OFFSETS[0] * _edge(tris), band != 0)
    assert np.array_equal((w > 0.5)[keep], (w64 > 0.5)[keep]), f"{what}: contains differs from float64 on {int(((w > 0.5) != (w64 > 0.5))[keep].sum())}"
    err = np.abs(w.astype(np.float64) - w64)
    rows = []
    for b in sorted(set(band[~np.isnan(band)].tolist())) + [np.nan]:
        m = np.isnan(band) if np.isnan(b) else band == b
        rows.append(f"{'uniform' if np.isnan(b) else ('vertex' if b == 0 else f'{b:+g}')}: {err[m].max():.3g}")
    print(f"{what}: max |w - w64| per band: " + ", ".join(rows))
    assert err[band != 0].max() <= bound, what


@pytest.mark.gpu
@pytest.mark.parametrize("n", [10_000, 100_000])
def test_fast_mesh_against_float64(ctx, n):
    tris = _torus(n, 4)
    pts, band = _points(tris, np.random.default_rng(62), 64 if n > 10_000 else 512, 512 if n > 10_000 else 4096)
    s = ctx.upload(_flat(tris, True))
    try:
        w = s.winding_numbers(_t(pts)).cpu().numpy()
        assert np.array_equal(s.contains(_t(pts)).cpu().numpy(), w > 0.5)
        assert np.array_equal(w.view(np.uint32), s.winding_numbers(_t(pts), beta=2.0).cpu().numpy().view(np.uint32))
        _classify(s, tris, pts, band, w, f"torus {n}")
    finally:
        s.close()


@pytest.mark.gpu
def test_open_soup_gives_fractional_winding(ctx):
    tris = _half(_torus(10_000, 4))
    pts, band = _points(tris, np.random.default_rng(63), 256, 4096)
    s = ctx.upload(_flat(tris, True))
    try:
        w64 = _w64(tris, pts)
        assert np.sum((w64 > 0.1) & (w64 < 0.9)) > len(pts) // 10  # fractional values, not a closed surface
        for beta in (2.0, INF):
            w = s.winding_numbers(_t(pts), beta=beta).cpu().numpy()
            err = np.abs(w.astype(np.float64) - w64)[band != 0]
            print(f"half torus, beta {beta}: max |w - w64| {err.max():.3g}")
            assert err.max() <= OPEN_BOUND[beta]
    finally:
        s.close()


# ---- signed distance ----------------------------------------------------------------------------
@pytest.mark.gpu
def test_signed_distance(ctx):
    import torch
    tris = _torus(10_000, 5)
    pts, _ = _points(tris, np.random.default_rng(64), 512, 4096)
    s = ctx.upload(_flat(tris, True))
    try:
        pt = _t(pts)
        for max_dist in (None, 0.5, torch.full((len(pts),), 2.0, device="cuda:0")):
            sd, hid, pos, nrm = s.signed_distance(pt, max_dist=max_dist)
            ref = s.closest_points(pt, max_dist=max_dist)
            ins = s.contains(pt).cpu().numpy()
            sd, hid_r, dist = sd.cpu().numpy(), ref[0].cpu().numpy(), ref[1].cpu().numpy()
            assert np.array_equal(hid.cpu().numpy(), hid_r) and torch.equal(pos, ref[2]) and torch.equal(nrm, ref[3])
            hit = hid_r >= 0
            assert np.array_equal(np.abs(sd[hit]).view(np.uint32), dist[hit].view(np.uint32))
            assert np.array_equal(np.signbit(sd), ins)
            assert np.all(np.isinf(sd[~hit]))
            if max_dist is not None:
                assert (~hit).sum() > 100 and ins[~hit].any() and (~ins[~hit]).any()
    finally:
        s.close()


# ---- moments and updates ------------------------------------------------------------------------
@pytest.mark.gpu
def test_moments_are_deterministic_and_sized_per_node_slot(ctx, host_model):
    tris = _ball()
    n = len(tris)
    flat = _flat_records(tris, [(rtb200.PRIM_TRIANGLES, 0, 300)] + [(rtb200.PRIM_MESH, a, c) for a, c in _overlap_layout(n)[1:]])
    a, b = ctx.upload(flat), ctx.upload(flat)
    twin = ctx.upload(_run_twin(flat))
    try:
        dev, up = a.device_bytes, a.upload_bytes
        a.mesh_moments()
        assert a.device_bytes - dev == 64 * sum(c for _, c in _overlap_layout(n)[1:]) and a.upload_bytes == up
        a.mesh_moments()  # a second call does nothing
        assert a.device_bytes - dev == 64 * sum(c for _, c in _overlap_layout(n)[1:])
        pts, _ = _points(tris, np.random.default_rng(65), 512, 4096)
        pt = _t(pts)
        for beta in (1.0, 2.0, 4.0):
            assert np.array_equal(_bits(a.winding_numbers(pt, beta=beta)), _bits(b.winding_numbers(pt, beta=beta))), beta
        # overlapping records each count: the exact sum equals the run twin's within the summation bound
        w_mesh = a.winding_numbers(pt, beta=INF).cpu().numpy().astype(np.float64)
        w_twin = twin.winding_numbers(pt).cpu().numpy().astype(np.float64)
        assert np.abs(w_twin).max() > 1.5  # the enclosing records add up
        recs = _overlap_layout(n)
        abs_sum = sum(host_model(tris[a:a + c], pts)[1] for a, c in recs)
        assert np.all(np.abs(w_mesh - w_twin) <= sum(c for _, c in recs) * 2.0 ** -23 * abs_sum)
    finally:
        for x in (a, b, twin):
            x.close()


@pytest.mark.gpu
@pytest.mark.parametrize("refit", [False, True])
def test_updates_keep_the_moments_current(ctx, refit):
    tris = _torus(100_000, 7)
    new = twist(tris, 0.9, 1.05)
    s, fresh = ctx.upload(_flat(tris, True)), ctx.upload(_flat(new, True))
    try:
        pts, band = _points(new, np.random.default_rng(66), 64, 512)
        pt = _t(pts)
        s.winding_numbers(pt)  # builds the moments
        dev = s.device_bytes
        s.mesh_update(_t(new), refit=refit)
        assert s.device_bytes == dev
        w = s.winding_numbers(pt)
        if not refit:
            assert np.array_equal(_bits(w), _bits(fresh.winding_numbers(pt))), "rebuild differs from a fresh upload"
        else:
            _classify(s, new, pts, band, w.cpu().numpy(), "refit twist")
    finally:
        s.close()
        fresh.close()


# ---- streams ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("where", ["side", "default"])
def test_points_from_torch_on_a_stream(ctx, where):
    import torch
    tris = _torus(1_000_000, 6)
    s = ctx.upload(_flat(tris, True, lead_sphere=False))
    try:
        s.mesh_moments()
        torch.cuda.synchronize()
        st = torch.cuda.Stream(device=0) if where == "side" else torch.cuda.default_stream(0)
        with torch.cuda.stream(st):
            pts = _torch_points(tris, 1 << 20, 7)
            for _ in range(4):  # work ahead of the query: a missing wait would read unfinished points
                pts = (pts * 1.0001).contiguous()
            exp_pts = pts.clone()
            got = s.winding_numbers(pts)
            ins = s.contains(pts)
            pts.fill_(float("nan"))
        torch.cuda.synchronize()
        exp = s.winding_numbers(exp_pts)
        assert torch.equal(got, exp) and torch.equal(ins, exp > 0.5)
        assert int(ins.sum()) > 1000
    finally:
        s.close()


@pytest.mark.gpu
def test_query_does_not_synchronise(ctx):
    import torch
    tris = _torus(100_000, 5)
    s = ctx.upload(_flat(tris, True, lead_sphere=False))
    try:
        pts = _torch_points(tris, 4096, 8)
        ref = s.winding_numbers(pts)
        torch.cuda.synchronize()
        st = torch.cuda.Stream(device=0)
        with torch.cuda.stream(st):
            torch.cuda._sleep(1_000_000_000)  # about half a second
            got = s.winding_numbers(pts)
            ins = s.contains(pts)
        busy = not st.query()
        st.synchronize()
        assert busy, "the query call waited for its stream"
        assert torch.equal(got, ref) and torch.equal(ins, ref > 0.5)
    finally:
        s.close()


@pytest.mark.gpu
def test_a_later_update_waits_for_the_query(ctx):
    import torch
    tris = _torus(1_000_000, 6)
    new = twist(tris, 0.6, 1.05)
    s = ctx.upload(_flat(tris, True, lead_sphere=False))
    old_ref, new_ref = ctx.upload(_flat(tris, True, lead_sphere=False)), ctx.upload(_flat(new, True, lead_sphere=False))
    try:
        pts = _torch_points(tris, 1 << 21, 9)
        rec = _t(new)
        s.mesh_moments()
        torch.cuda.synchronize()
        sa, sb = torch.cuda.Stream(device=0), torch.cuda.Stream(device=0)
        with torch.cuda.stream(sa):
            torch.cuda._sleep(200_000_000)  # the query is still queued when the update is enqueued
            before = s.winding_numbers(pts)
        with torch.cuda.stream(sb):
            s.mesh_update(rec)
        with torch.cuda.stream(sa):
            after = s.winding_numbers(pts)
        torch.cuda.synchronize()
        assert torch.equal(before, old_ref.winding_numbers(pts)), "the query before the update"
        assert torch.equal(after, new_ref.winding_numbers(pts)), "the query after the update"
        assert not torch.equal(before, after)
    finally:
        for x in (s, old_ref, new_ref):
            x.close()


@pytest.mark.gpu
def test_moments_follow_an_update_on_another_stream(ctx):
    """An update enqueued behind slow work on stream A, then the moments built from stream B: they are the new mesh's."""
    import torch
    tris = _torus(1_000_000, 6)
    new = twist(tris, 0.6, 1.05)
    s, ref = ctx.upload(_flat(tris, True, lead_sphere=False)), ctx.upload(_flat(new, True, lead_sphere=False))
    try:
        pts = _torch_points(tris, 1 << 16, 10)
        base = _t(new)
        torch.cuda.synchronize()
        sa, sb = torch.cuda.Stream(device=0), torch.cuda.Stream(device=0)
        with torch.cuda.stream(sa):
            torch.cuda._sleep(200_000_000)
            rec = (base * 1.0).contiguous()  # made on A, behind the sleep
            s.mesh_update(rec)
        with torch.cuda.stream(sb):
            s.mesh_moments()
            got = s.winding_numbers(pts)
        torch.cuda.synchronize()
        assert torch.equal(got, ref.winding_numbers(pts))
    finally:
        s.close()
        ref.close()


# ---- refusals -----------------------------------------------------------------------------------
def _raw(ctx, scene, n, pts, beta, w=None, ins=None, stream=None):
    p = lambda x: None if x is None else C.c_void_p(x if isinstance(x, int) else x.data_ptr())
    return ctx._lib.rtb_query_winding(ctx._h, scene._h, n, p(pts), beta, p(w), p(ins), p(stream))


@pytest.mark.gpu
def test_refused_calls_write_nothing(ctx):
    import torch
    tris = _ball()
    s, fresh = ctx.upload(_flat(tris, True)), ctx.upload(_flat(tris, True))
    try:
        s.mesh_moments()
        pts_np, _ = _points(tris, np.random.default_rng(67), 8, 0)
        n = len(pts_np)
        pts = _t(pts_np)
        w = torch.full((n,), 7.5, device="cuda:0")
        ins = torch.full((n,), 77, dtype=torch.uint8, device="cuda:0")
        mis = torch.zeros(n * 3 + 1, device="cuda:0", dtype=torch.float32)
        byte = mis.view(torch.uint8)
        host_w = np.full(n, 7.5, np.float32)
        host_ins = np.full(n, 77, np.uint8)
        pinned = rtb200.PinnedArray((n, 3))
        torch.cuda.synchronize()
        snap = (w.clone(), ins.clone())
        cases = {
            "n < 0": _raw(ctx, s, -1, pts, 2.0, w, ins),
            "beta NaN": _raw(ctx, s, n, pts, float("nan"), w, ins),
            "beta below 1": _raw(ctx, s, n, pts, 0.999, w, ins),
            "beta -inf": _raw(ctx, s, n, pts, -INF, w, ins),
            "no outputs": _raw(ctx, s, n, pts, 2.0),
            "mesh without moments": _raw(ctx, fresh, n, pts, 2.0, w, ins),
            "host points": _raw(ctx, s, n, np.ascontiguousarray(pts_np).ctypes.data, 2.0, w, ins),
            "no points": _raw(ctx, s, n, None, 2.0, w, ins),
            "misaligned points": _raw(ctx, s, n, byte[1:].data_ptr(), 2.0, w, ins),
            "misaligned winding": _raw(ctx, s, n, pts, 2.0, w.data_ptr() + 2, ins),
            "host winding": _raw(ctx, s, n, pts, 2.0, host_w.ctypes.data, ins),
            "host inside": _raw(ctx, s, n, pts, 2.0, w, host_ins.ctypes.data),
            "host inside only": _raw(ctx, s, n, pts, 2.0, None, host_ins.ctypes.data),
            "page-locked host inside": _raw(ctx, s, n, pts, 2.0, w, pinned._p.value),
        }
        torch.cuda.synchronize()
        pinned.close()
        for what, rc in cases.items():
            assert rc == ERR_INVALID, f"{what}: rc {rc}"
        assert torch.equal(w, snap[0]) and torch.equal(ins, snap[1]), "a refused call wrote its outputs"
        assert np.all(host_w == 7.5) and np.all(host_ins == 77)
        assert _raw(ctx, s, 0, None, 2.0, w) == 0  # n == 0: nothing to do
        assert _raw(ctx, fresh, n, pts, 2.0, w, ins) == ERR_INVALID
        assert "rtb_scene_mesh_moments" in ctx._lib.rtb_last_error(ctx._h).decode()
        nanp = _t(np.array([[np.nan, 0, 0]], np.float32))
        wn, inn = torch.zeros(1, device="cuda:0"), torch.ones(1, dtype=torch.uint8, device="cuda:0")
        assert _raw(ctx, s, 1, nanp, 2.0, wn, inn) == 0
        torch.cuda.synchronize()
        assert np.isnan(wn.item()) and inn.item() == 0  # a NaN point: NaN / outside
        with pytest.raises(rtb200.RtbError):
            s.winding_numbers(pts.cpu())
        with pytest.raises(rtb200.RtbError):
            s.winding_numbers(pts, beta=0.5)
        with pytest.raises(rtb200.RtbError):
            s.contains(pts, out=torch.zeros(n, dtype=torch.uint8, device="cuda:0"))
    finally:
        s.close()
        fresh.close()
