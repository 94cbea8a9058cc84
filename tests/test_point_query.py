"""rtb_query_points: the nearest point on the scene's TRIANGLES and MESH records within a strict per-point radius, and
proximity tests, on device buffers and ordered on the caller's stream (include/rtb.h, DESIGN 3e).  Oracles: the distance
function csrc/rtb_closest.h compiled for the host (a brute-force loop over it, and its CPU check against float64), and for
mesh records the run of the same triangles, which a mesh must reproduce bit for bit."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import rtb200
from rtb200 import PresetScene
from test_mesh import _ball, _flat, _flat_records, _preset3, _tris_from_facets
from test_mesh_update import _overlap_layout, twist
from test_ray_query import _run_twin

ERR_INVALID = -1
CSRC = os.path.join(rtb200.PKG, "csrc")


# ---- host side (no device) --------------------------------------------------------------------
def test_closest_point_check_on_the_cpu(tmp_path):
    """csrc/rtb_closest.h for the host over random and adversarial (point, triangle) pairs: q inside the leaf box, the pruning
    lemma boxDist2 <= d2, finite outputs, and the distance within the stated bound of a float64 closest point."""
    exe = str(tmp_path / "closest_point_check")
    src = os.path.join(rtb200.ROOT, "tests", "closest_point_check.cpp")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-o", exe, src])
    for seed in (1, 2):
        out = subprocess.run([exe, str(seed), "200000"], capture_output=True, text=True)
        print(out.stdout)
        assert out.returncode == 0, out.stdout
        counts = dict(re.findall(r"(\w+) (\d+)", out.stdout.splitlines()[-1]))
        assert int(counts["violations"]) == 0 and int(counts["checked"]) == 200000
        assert int(counts["zero_cross"]) > 10000 and int(counts["on_vertex"]) > 10000 and int(counts["in_plane"]) > 10000


def test_header_point_query_matches_the_bindings():
    text = open(os.path.join(rtb200.ROOT, "include", "rtb.h")).read()
    assert re.search(r"enum \{ RTB_QUERY_CLOSEST = 0, RTB_QUERY_ANY = 1 \};", text)
    assert re.search(r"int rtb_query_points\(rtb_ctx \*ctx, const rtb_scene \*scene, int64_t n, const float \*points, "
                     r"const float \*rmax, float rmax_all,\s+int32_t flags, int32_t \*hit_id, float \*distance, float \*position, "
                     r"float \*normal, uint8_t \*near,\s+void \*stream\);", text)
    assert (rtb200.QUERY_CLOSEST, rtb200.QUERY_ANY) == (0, 1)
    assert "rtb_query_points" in rtb200.ABI_SYMBOLS
    assert "#define RTB_ABI_VERSION 5" in text


# ---- host model: the header compiled into a small library --------------------------------------
_HOST_SRC = r"""
#include "rtb_closest.h"
// brute force over packed records t[m][12] (a, a - b, a - c, n) as one TRIANGLES run with ids base + k
extern "C" void closest_all(const float *t, int m, int base, const float *pts, long n, const float *rmax, int *id, float *dist,
                            float *pos, float *nrm)
{
    for (long i = 0; i < n; i++)
    {
        const float *p = pts + 3 * i;
        const float r = rmax[i];
        float best = r * r, q[3], bq[3] = {0, 0, 0};
        int k = -1;
        if (r > 0.0f && p[0] == p[0] && p[1] == p[1] && p[2] == p[2])
            for (int j = 0; j < m; j++)
            {
                const float d2 = rtb_closest::closestPoint(p, t + 12 * (long)j, q);
                if (d2 < best) { best = d2; k = j; bq[0] = q[0]; bq[1] = q[1]; bq[2] = q[2]; }
            }
        id[i] = k >= 0 ? base + k : -1;
        dist[i] = k >= 0 ? sqrtf(best) : -1.0f;
        for (int c = 0; c < 3; c++) { pos[3 * i + c] = bq[c]; nrm[3 * i + c] = k >= 0 ? t[12 * (long)k + 9 + c] : 0.0f; }
    }
}
"""


@pytest.fixture(scope="module")
def host_model(tmp_path_factory):
    d = tmp_path_factory.mktemp("closest_host")
    src, so = d / "closest_host.cpp", d / "closest_host.so"
    src.write_text(_HOST_SRC)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-I", CSRC, "-o", str(so), str(src)])
    lib = C.CDLL(str(so))
    vp = C.c_void_p
    lib.closest_all.argtypes = [vp, C.c_int, C.c_int, vp, C.c_long, vp, vp, vp, vp, vp]

    def run(tris, pts, rmax=np.inf, base=0):
        packed = _packed(tris)
        pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 3)
        n = len(pts)
        r = np.ascontiguousarray(np.broadcast_to(np.float32(rmax), (n,)), np.float32)
        out = (np.zeros(n, np.int32), np.zeros(n, np.float32), np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32))
        lib.closest_all(packed.ctypes.data, len(packed), base, pts.ctypes.data, n, r.ctypes.data, *(o.ctypes.data for o in out))
        return out
    return run


def _packed(tris):
    """loose records (a, b, c, n) -> the packed stream's record (a, a - b, a - c, n), as k_pack_triangles writes it"""
    t = np.ascontiguousarray(tris, np.float32).reshape(-1, 12)
    return np.ascontiguousarray(np.concatenate([t[:, 0:3], t[:, 0:3] - t[:, 3:6], t[:, 0:3] - t[:, 6:9], t[:, 9:12]], 1), np.float32)


def _dist64(tris, pts):
    """float64 distance from every point to the nearest triangle (brute force, numpy)"""
    v = np.asarray(tris, np.float64)[:, :9].reshape(-1, 3, 3)
    a, b, c = v[:, 0], v[:, 1], v[:, 2]
    out = np.empty(len(pts))
    for i, p in enumerate(np.asarray(pts, np.float64)):
        def seg(s0, s1):
            d = s1 - s0
            dd = np.einsum("ij,ij->i", d, d)
            t = np.clip(np.where(dd > 0, np.einsum("ij,ij->i", p - s0, d) / np.where(dd > 0, dd, 1), 0), 0, 1)
            r = p - (s0 + d * t[:, None])
            return np.sqrt(np.einsum("ij,ij->i", r, r))
        best = np.minimum(seg(a, b), np.minimum(seg(a, c), seg(b, c)))
        n = np.cross(b - a, c - a)
        nn = np.einsum("ij,ij->i", n, n)
        ok = nn > 0
        h = np.einsum("ij,ij->i", p - a, n) / np.where(ok, nn, 1)
        q = p - n * h[:, None]
        ins = ok & (np.einsum("ij,ij->i", np.cross(b - a, q - a), n) >= 0) & (np.einsum("ij,ij->i", np.cross(c - b, q - b), n) >= 0) \
            & (np.einsum("ij,ij->i", np.cross(a - c, q - c), n) >= 0)
        best = np.where(ins, np.minimum(best, np.abs(h) * np.sqrt(nn)), best)
        out[i] = best.min()
    return out


# ---- points -----------------------------------------------------------------------------------
def _points(tris, rng, n, centre=None):
    """near the surface (both sides), far away, uniform in the box (inside a torus' tube too), exactly on vertices, and --
    for a torus -- around its centre, where many triangles are almost equally near"""
    v = tris[:, :9].reshape(-1, 3, 3).astype(np.float64)
    lo, hi = v.reshape(-1, 3).min(0), v.reshape(-1, 3).max(0)
    ext = float(np.max(hi - lo))
    k = rng.integers(0, len(tris), n)
    surf = np.einsum("ni,nij->nj", rng.dirichlet([1, 1, 1], n), v[k])
    nrm = np.cross(v[k, 1] - v[k, 0], v[k, 2] - v[k, 0])
    nrm /= np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-30)
    parts = [surf + nrm * rng.uniform(-0.01, 0.01, (n, 1)) * ext,
             (lo + hi) / 2 + rng.normal(size=(n, 3)) * ext * 2,
             lo + rng.uniform(size=(n, 3)) * (hi - lo),
             v[k, rng.integers(0, 3, n)]]
    if centre is not None:
        parts.append(np.asarray(centre) + rng.normal(size=(n, 3)) * 1e-3)
        parts.append(np.tile(np.asarray(centre, np.float64), (4, 1)))
    return np.ascontiguousarray(np.concatenate(parts), np.float32)


def _torus(n, seed):
    return _tris_from_facets(rtb200.torus_triangles(n, seed=seed))


TORUS_CENTRE = (0.0, 16.0, 0.0)  # torus_triangles' default centre


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


def _np(res):
    return tuple(x.cpu().numpy() for x in res)


def _same(a, b):
    """per-point bitwise equality of two closest results"""
    eq = (a[0] == b[0]) & (a[1].view(np.uint32) == b[1].view(np.uint32))
    return eq & np.all(a[2].view(np.uint32) == b[2].view(np.uint32), 1) & np.all(a[3].view(np.uint32) == b[3].view(np.uint32), 1)


def _d2(pts, pos):
    """the winner's squared distance, recomputed from its closest point in the contract's float32 order"""
    d = (np.asarray(pts, np.float32) - pos).astype(np.float32)
    return ((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]).astype(np.float32) + d[:, 2] * d[:, 2]).astype(np.float32)


def _masked(res, pts, rmax):
    """unbounded results with every winner at d2 >= fl(r * r) (or r NaN / <= 0) turned into a miss"""
    hid, dist, pos, nrm = (x.copy() for x in res)
    r = np.broadcast_to(np.float32(rmax), hid.shape).astype(np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        keep = (hid >= 0) & (r > 0) & (_d2(pts, pos) < (r * r).astype(np.float32))
    hid[~keep], dist[~keep] = -1, -1
    pos[~keep], nrm[~keep] = 0, 0
    return hid, dist, pos, nrm


def _radii(dist, rng):
    """per-point radii around the unbounded distance (-1 = miss): exactly it, its neighbours, half, double, special values"""
    n = len(dist)
    dd = np.where(dist >= 0, dist, np.float32(rng.uniform(1, 100))).astype(np.float32)
    table = [dd, np.nextafter(dd, np.float32(np.inf)), np.nextafter(dd, np.float32(-np.inf)), dd / 2, dd * 2,
             np.zeros(n, np.float32), np.full(n, -1, np.float32), np.full(n, np.nan, np.float32), np.full(n, np.inf, np.float32),
             (rng.uniform(0, 2, n) * dd).astype(np.float32)]
    kind = rng.integers(0, len(table), n)
    b = np.empty(n, np.float32)
    for k, v in enumerate(table):
        b[kind == k] = v[kind == k]
    return b


@pytest.fixture(scope="module")
def ctx():
    c = rtb200.Context(0)
    yield c
    c.close()


# ---- mesh == run, bit for bit -----------------------------------------------------------------
def _special():
    ball = _ball()
    dup = np.concatenate([ball, ball[::-1], ball])  # ties go to the lowest index
    zero = ball.copy()
    zero[::7, 3:6] = zero[::7, 0:3]  # a collapsed vertex
    zero[3::11, 3:9] = np.tile(zero[3::11, 0:3], 2)  # three equal vertices
    coll = ball.copy()
    coll[5::9, 6:9] = coll[5::9, 0:3] + (coll[5::9, 3:6] - coll[5::9, 0:3]) * np.float32(2.5)  # collinear
    g = np.linspace(-10, 10, 41, dtype=np.float32)
    x, y = np.meshgrid(g, g, indexing="ij")
    q = np.stack([x, y, np.zeros_like(x)], -1)
    a, b, c, d = q[:-1, :-1], q[1:, :-1], q[1:, 1:], q[:-1, 1:]
    plate_v = np.concatenate([np.stack([a, b, c], -2).reshape(-1, 9), np.stack([a, c, d], -2).reshape(-1, 9)])
    plate = np.concatenate([plate_v, np.tile([0, 0, 1], (len(plate_v), 1))], 1).astype(np.float32)  # coplanar: many ties
    far = ball.copy()
    far[:, :9] += np.float32(1e4)
    return np.concatenate([dup, zero, coll, plate, far])


CASES = ["ball", "torus100k", "torus1m", "special", "overlap", "mixed"]


def _case(name):
    """(mesh scene, triangles to place points around, torus centre or None, points per set)"""
    if name == "ball":
        return _preset3(True), _ball(), None, 1024
    if name.startswith("torus"):
        tris = _torus(100_000 if name == "torus100k" else 1_000_000, 5 if name == "torus100k" else 6)
        return _flat(tris, True), tris, TORUS_CENTRE, 2048 if name == "torus100k" else 818  # 1 M: 5 x 818 + 4 = 4094 points
    if name == "special":
        tris = _special()
        return _flat(tris, True), tris, None, 2048
    tris = _ball()
    if name == "overlap":
        return _flat_records(tris, [(rtb200.PRIM_TRIANGLES, 0, 300)] + [(rtb200.PRIM_MESH, a, c) for a, c in _overlap_layout(len(tris))[1:]]), \
            tris, None, 1024
    return _flat_records(tris, [(rtb200.PRIM_MESH, 0, 400), (rtb200.PRIM_TRIANGLES, 200, len(tris) - 200)]), tris, None, 1024


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_mesh_equals_run(ctx, name):
    """Every mesh query -- unbounded, bounded per point, one radius for all, any -- equals the run's bit for bit; bounded ==
    the masked unbounded result; any == the bounded closest query hits."""
    scene, tris, centre, n = _case(name)
    flat = scene.flat if hasattr(scene, "flat") else scene
    sm, sr = ctx.upload(flat), ctx.upload(_run_twin(flat))
    try:
        rng = np.random.default_rng(51)
        pts = _points(tris, rng, n, centre)
        pt = _t(pts)
        full = _np(sm.closest_points(pt))
        assert _same(full, _np(sr.closest_points(pt))).all(), f"{name}: mesh differs from the run"
        assert (full[0] >= 0).all() and np.isfinite(full[1]).all()
        assert _same(_np(sm.closest_points(pt, max_dist=float("inf"))), full).all()
        for rep in range(2):
            r = _radii(full[1], rng)
            exp = _masked(full, pts, r)
            for s in (sm, sr):
                got = _np(s.closest_points(pt, max_dist=_t(r)))
                assert _same(got, exp).all(), f"{name}: the bounded query differs from the masked one on {int((~_same(got, exp)).sum())}"
                near = s.closest_points(pt, max_dist=_t(r), any_hit=True).cpu().numpy()
                assert near.dtype == np.bool_ and np.array_equal(near, exp[0] >= 0), f"{name}: any differs from the bounded hits"
        for r in (0.0, -1.0, float("nan"), 0.5, 5.0):
            exp = _masked(full, pts, r)
            for s in (sm, sr):
                assert _same(_np(s.closest_points(pt, max_dist=r)), exp).all(), f"{name}: max_dist={r}"
                assert np.array_equal(s.closest_points(pt, max_dist=r, any_hit=True).cpu().numpy(), exp[0] >= 0)
        print(f"{name}: {len(pts)} points, mesh == run")
    finally:
        sm.close()
        sr.close()
        if hasattr(scene, "close"):
            scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ball", "torus100k", "special"])
def test_gpu_equals_host_and_float64(ctx, host_model, name):
    """The GPU answer equals a brute-force loop over the host-compiled header bit for bit, and lies within the header's stated
    bound of the float64 distance."""
    scene, tris, centre, _ = _case(name)
    flat = scene.flat if hasattr(scene, "flat") else scene
    s = ctx.upload(flat)
    try:
        pts = _points(tris, np.random.default_rng(52), 64, centre)
        f = flat.contents if hasattr(flat, "contents") else flat
        base = next(int(f.prims[i].base_id) for i in range(f.n_prims) if f.prims[i].type == rtb200.PRIM_MESH)
        got = _np(s.closest_points(_t(pts)))
        host = host_model(tris, pts, base=base)
        assert _same(got, host).all(), f"{name}: GPU differs from the host model on {int((~_same(got, host)).sum())} points"
        r = np.float32(2.0)
        assert _same(_np(s.closest_points(_t(pts), max_dist=float(r))), host_model(tris, pts, r, base)).all()
        ref = _dist64(tris, pts)
        mag = np.abs(pts).max(1).astype(np.float64)
        a = tris[got[0] - base, 0:3].astype(np.float64)
        ext = np.ptp(tris[:, :9].reshape(-1, 3, 3), axis=1).max(1)[got[0] - base].astype(np.float64)
        bound = 1e-4 * (np.linalg.norm(pts - a, axis=1) + ext) + 8 * mag * 2.0 ** -24
        err = np.abs(got[1].astype(np.float64) - ref)
        print(f"{name}: worst |d - d64| {err.max():.3g}")
        assert (err <= bound).all()
    finally:
        s.close()
        if hasattr(scene, "close"):
            scene.close()


# ---- records outside the query ---------------------------------------------------------------
def _with_mesh(flat, tris):
    """the flat scene with one MESH record of `tris` appended (after its own records; its loose triangles kept)"""
    f = rtb200.FlatScene.from_buffer_copy(flat.contents)
    prims = (rtb200.Prim * (f.n_prims + 1))()
    C.memmove(prims, f.prims, C.sizeof(rtb200.Prim) * f.n_prims)
    old = np.ctypeslib.as_array(f.loose_tri, shape=(f.n_loose, 12)).copy() if f.n_loose else np.zeros((0, 12), np.float32)
    loose = np.ascontiguousarray(np.concatenate([old, tris]), np.float32)
    p = prims[f.n_prims]
    p.type, p.material, p.base_id, p.first, p.count = rtb200.PRIM_MESH, 0, f.n_top, len(old), len(tris)
    f.n_prims, f.prims = f.n_prims + 1, prims
    f.n_loose, f.loose_tri = len(loose), loose.ctypes.data_as(C.POINTER(C.c_float))
    f.n_top += len(tris)
    f._keep = (prims, loose, flat)
    return f, int(p.base_id)


@pytest.mark.gpu
@pytest.mark.parametrize("preset", [2, 5])
def test_planes_spheres_and_the_tunnel_are_ignored(ctx, preset):
    s = PresetScene(5, "sah", 24) if preset == 5 else PresetScene(2)
    tris = twist(_ball(), 0.3)
    only = ctx.upload(_flat(tris, True, lead_sphere=False))
    plain = ctx.upload(s.flat)
    f, base = _with_mesh(s.flat, tris)
    both = ctx.upload(f)
    try:
        v = tris[:, :9].reshape(-1, 3)
        pts = _points(tris, np.random.default_rng(53), 512)
        pts = np.concatenate([pts, (v.min(0) + np.random.default_rng(54).uniform(size=(512, 3)) * (v.max(0) - v.min(0) + 200) - 100)
                              .astype(np.float32)])
        pt = _t(pts)
        miss = _np(plain.closest_points(pt))
        assert (miss[0] == -1).all() and (miss[1] == -1).all() and not miss[2].any() and not miss[3].any()
        assert not plain.closest_points(pt, any_hit=True).cpu().numpy().any()
        ref, got = _np(only.closest_points(pt)), _np(both.closest_points(pt))
        got = (np.where(got[0] >= 0, got[0] - base, -1).astype(np.int32),) + got[1:]
        assert _same(got, ref).all()
        assert np.array_equal(both.closest_points(pt, max_dist=3.0, any_hit=True).cpu().numpy(),
                              only.closest_points(pt, max_dist=3.0, any_hit=True).cpu().numpy())
    finally:
        for x in (only, plain, both):
            x.close()
        s.close()


# ---- tree independence -------------------------------------------------------------------------
@pytest.mark.gpu
def test_refit_rebuild_and_fresh_upload_answer_alike(ctx):
    """After mesh_update from a CUDA tensor on a side stream, with the query enqueued right behind it and no host synchronise,
    a refitted tree, a rebuilt tree and a fresh upload of the new triangles answer bit for bit alike."""
    import torch
    tris = _torus(200_000, 7)
    new = twist(tris, 0.9, 1.05)
    pts = _t(_points(new, np.random.default_rng(55), 4096, TORUS_CENTRE))
    r = torch.full((pts.shape[0],), 0.3, device="cuda:0")
    refit, rebuild = ctx.upload(_flat(tris, True)), ctx.upload(_flat(tris, True))
    fresh = ctx.upload(_flat(new, True))
    try:
        torch.cuda.synchronize()
        st = torch.cuda.Stream(device=0)
        res = {}
        with torch.cuda.stream(st):
            rec = _t(new)
            for s, is_refit, key in ((refit, True, "refit"), (rebuild, False, "rebuild")):
                s.mesh_update(rec, refit=is_refit)
                res[key] = (s.closest_points(pts), s.closest_points(pts, max_dist=r), s.closest_points(pts, max_dist=r, any_hit=True))
        res["fresh"] = (fresh.closest_points(pts), fresh.closest_points(pts, max_dist=r), fresh.closest_points(pts, max_dist=r, any_hit=True))
        torch.cuda.synchronize()
        ref = res["fresh"]
        for key in ("refit", "rebuild"):
            assert _same(_np(res[key][0]), _np(ref[0])).all() and _same(_np(res[key][1]), _np(ref[1])).all(), key
            assert torch.equal(res[key][2], ref[2]), key
    finally:
        for s in (refit, rebuild, fresh):
            s.close()


# ---- streams -----------------------------------------------------------------------------------
def _torch_points(tris, n, seed):
    """points made by torch ops on the current stream: uniform in the model's box, grown by a quarter"""
    import torch
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    v = torch.from_numpy(tris[:, :9].reshape(-1, 3)).to("cuda:0")
    lo, hi = v.min(0).values, v.max(0).values
    return (lo - (hi - lo) / 8 + torch.rand(n, 3, device="cuda:0", generator=g) * (hi - lo) * 1.25).contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["side", "default"])
def test_points_from_torch_on_a_stream(ctx, where):
    import torch
    tris = _torus(1_000_000, 6)
    s = ctx.upload(_flat(tris, True, lead_sphere=False))
    try:
        torch.cuda.synchronize()
        st = torch.cuda.Stream(device=0) if where == "side" else torch.cuda.default_stream(0)
        with torch.cuda.stream(st):
            pts = _torch_points(tris, 1 << 20, 7)
            for _ in range(4):  # work ahead of the query: a missing wait would read unfinished points
                pts = (pts * 1.0001).contiguous()
            rmax = (pts[:, 0].abs() * 0.1 + 0.5).contiguous()
            exp_pts, exp_r = pts.clone(), rmax.clone()
            got = s.closest_points(pts, max_dist=rmax)
            near = s.closest_points(pts, max_dist=rmax, any_hit=True)
            pts.fill_(float("nan"))
            rmax.fill_(0.0)
        torch.cuda.synchronize()
        exp = s.closest_points(exp_pts, max_dist=exp_r)
        assert all(torch.equal(a, b) for a, b in zip(got, exp))
        assert torch.equal(near, exp[0] >= 0)
        assert int((exp[0] >= 0).sum()) > 1000
    finally:
        s.close()


@pytest.mark.gpu
def test_query_does_not_synchronise(ctx):
    import torch
    tris = _torus(100_000, 5)
    s = ctx.upload(_flat(tris, True, lead_sphere=False))
    try:
        pts = _torch_points(tris, 4096, 8)
        ref = s.closest_points(pts)
        torch.cuda.synchronize()
        st = torch.cuda.Stream(device=0)
        with torch.cuda.stream(st):
            torch.cuda._sleep(1_000_000_000)  # about half a second
            got = s.closest_points(pts)
            near = s.closest_points(pts, max_dist=1.0, any_hit=True)
        busy = not st.query()
        st.synchronize()
        assert busy, "the query call waited for its stream"
        assert all(torch.equal(a, b) for a, b in zip(got, ref))
        assert np.array_equal(near.cpu().numpy(), _masked(_np(ref), pts.cpu().numpy(), 1.0)[0] >= 0)
    finally:
        s.close()


@pytest.mark.gpu
def test_a_later_update_waits_for_the_query(ctx):
    """A large query on stream A, then an update on stream B: the query sees the old triangles, a later one the new."""
    import torch
    tris = _torus(1_000_000, 6)
    new = twist(tris, 0.6, 1.05)
    s = ctx.upload(_flat(tris, True, lead_sphere=False))
    old_ref, new_ref = ctx.upload(_flat(tris, True, lead_sphere=False)), ctx.upload(_flat(new, True, lead_sphere=False))
    try:
        pts = _torch_points(tris, 1 << 21, 9)
        rec = _t(new)
        torch.cuda.synchronize()
        sa, sb = torch.cuda.Stream(device=0), torch.cuda.Stream(device=0)
        with torch.cuda.stream(sa):
            torch.cuda._sleep(200_000_000)  # the query is still queued when the update is enqueued
            before = s.closest_points(pts)
        with torch.cuda.stream(sb):
            s.mesh_update(rec)
        with torch.cuda.stream(sa):
            after = s.closest_points(pts)
        torch.cuda.synchronize()
        assert all(torch.equal(g, e) for g, e in zip(before, old_ref.closest_points(pts))), "the query before the update"
        assert all(torch.equal(g, e) for g, e in zip(after, new_ref.closest_points(pts))), "the query after the update"
        assert not torch.equal(before[1], after[1])
    finally:
        for x in (s, old_ref, new_ref):
            x.close()


# ---- refusals ----------------------------------------------------------------------------------
def _raw(ctx, scene, n, pts, rmax, flags, hid=None, dist=None, pos=None, nrm=None, near=None, stream=None):
    p = lambda x: None if x is None else C.c_void_p(x if isinstance(x, int) else x.data_ptr())
    return ctx._lib.rtb_query_points(ctx._h, scene._h, n, p(pts), p(rmax), float("inf"), flags, p(hid), p(dist), p(pos), p(nrm),
                                     p(near), p(stream))


@pytest.mark.gpu
def test_refused_calls_write_nothing(ctx):
    import torch
    tris = _ball()
    s = ctx.upload(_flat(tris, True))
    try:
        pts_np = _points(tris, np.random.default_rng(56), 64)
        n = len(pts_np)
        pts = _t(pts_np)
        rmax = torch.full((n,), 100.0, device="cuda:0")
        hid = torch.full((n,), 12345, dtype=torch.int32, device="cuda:0")
        dist = torch.full((n,), 7.5, device="cuda:0")
        pos = torch.full((n, 3), 7.5, device="cuda:0")
        nrm = torch.full((n, 3), 7.5, device="cuda:0")
        near = torch.full((n,), 77, dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()
        snap = [x.clone() for x in (hid, dist, pos, nrm, near)]
        CL, ANY = rtb200.QUERY_CLOSEST, rtb200.QUERY_ANY
        host = np.ascontiguousarray(pts_np)
        pinned = rtb200.PinnedArray((n, 3))
        pinned.array[:] = pts_np
        mis = torch.zeros(n * 3 + 1, device="cuda:0", dtype=torch.float32)
        byte = mis.view(torch.uint8)
        torch.cuda.synchronize()
        cases = {
            "host points": _raw(ctx, s, n, host.ctypes.data, None, CL, hid, dist, pos, nrm),
            "page-locked host points": _raw(ctx, s, n, pinned._p.value, None, CL, hid, dist, pos, nrm),
            "host rmax": _raw(ctx, s, n, pts, np.full(n, 5, np.float32).ctypes.data, CL, hid, dist, pos, nrm),
            "misaligned points": _raw(ctx, s, n, byte[1:].data_ptr(), None, CL, hid, dist, pos, nrm),
            "no points": _raw(ctx, s, n, None, None, CL, hid, dist, pos, nrm),
            "n < 0": _raw(ctx, s, -1, pts, None, CL, hid, dist, pos, nrm),
            "unknown flags": _raw(ctx, s, n, pts, None, 2, hid, dist, pos, nrm),
            "ANY with closest outputs": _raw(ctx, s, n, pts, rmax, ANY, hid, near=near),
            "ANY without near": _raw(ctx, s, n, pts, rmax, ANY),
            "CLOSEST with near": _raw(ctx, s, n, pts, rmax, CL, hid, dist, pos, nrm, near),
            "misaligned output": _raw(ctx, s, n, pts, rmax, CL, dist.data_ptr() + 2),
        }
        torch.cuda.synchronize()
        pinned.close()
        for what, rc in cases.items():
            assert rc == ERR_INVALID, f"{what}: rc {rc}"
        for a, b in zip((hid, dist, pos, nrm, near), snap):
            assert torch.equal(a, b), "a refused call wrote its outputs"
        assert _raw(ctx, s, 0, None, None, CL) == 0  # n == 0: nothing to do
        with pytest.raises(rtb200.RtbError):
            s.closest_points(pts.cpu())
        with pytest.raises(rtb200.RtbError):
            s.closest_points(pts, max_dist=rmax[:-1])
        with pytest.raises(rtb200.RtbError):
            s.closest_points(pts[:, :2].contiguous())
    finally:
        s.close()
