"""rtb_query_rays: closest hits under a strict per-ray bound and occlusion tests, on device buffers and ordered on the caller's
stream (include/rtb.h).  The oracles are the host-array path rtb_intersect_rays, masked by the bound, and for mesh records
the run of the same triangles (a mesh may differ from it only where the run's winning pair lies in the grazing band of
csrc/rtb_bvh.h, checked here on the CPU)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import rtb200
from rtb200 import PresetScene
from test_mesh import _ball, _flat, _flat_records, _in_grazing_band, _preset3, _ray_sets, _tris_from_facets
from test_mesh_update import _overlap_layout, twist

ERR_INVALID = -1
FLT_MAX = np.float32(3.4028235e38)


@pytest.fixture(scope="module")
def ctx():
    c = rtb200.Context(0)
    yield c
    c.close()


# ---- scenes and rays ----------------------------------------------------------------------------
def _camera_rays(cam, w, h):
    """The primary rays of a w x h frame, built on the host as Camera.cpp:20-26 does (test_gpu_parity)."""
    xs, ys = np.meshgrid(np.arange(w, dtype=np.float32), np.arange(h, dtype=np.float32))
    d = np.float32(1.0) / np.float32(h)
    sx, sy = (xs + np.float32(0.5)) * d, np.float32(1) - (ys + np.float32(0.5)) * d
    right, up, front = (np.array(v, np.float32) for v in (cam.right, cam.up, cam.front))
    r = right[None, None, :] * ((sx - np.float32(cam.xcenter)) * np.float32(cam.fov_scale))[..., None]
    u = up[None, None, :] * ((sy - np.float32(0.5)) * np.float32(cam.fov_scale))[..., None]
    v = front[None, None, :] + r + u
    dirs = v * (np.float32(1) / np.sqrt(v[..., 0] * v[..., 0] + v[..., 1] * v[..., 1] + v[..., 2] * v[..., 2]))[..., None]
    eye = np.array(cam.eye, np.float32)
    return np.concatenate([np.broadcast_to(eye + dirs * np.float32(cam.forward), dirs.shape), dirs], 2).reshape(-1, 6).astype(np.float32)


def _loose_tris(flat):
    f = flat.contents if hasattr(flat, "contents") else flat
    return np.ctypeslib.as_array(f.loose_tri, shape=(f.n_loose, 12)).copy() if f.n_loose else np.zeros((0, 12), np.float32)


def _run_twin(flat):
    """The same flat scene with every MESH record turned into a TRIANGLES run (the mesh's oracle)."""
    f = rtb200.FlatScene.from_buffer_copy(flat.contents if hasattr(flat, "contents") else flat)
    prims = (rtb200.Prim * f.n_prims)()
    C.memmove(prims, f.prims, C.sizeof(rtb200.Prim) * f.n_prims)
    for p in prims:
        if p.type == rtb200.PRIM_MESH:
            p.type = rtb200.PRIM_TRIANGLES
    f.prims = prims
    f._keep = (prims, flat)
    return f


def _has_mesh(flat):
    f = flat.contents if hasattr(flat, "contents") else flat
    return any(f.prims[i].type == rtb200.PRIM_MESH for i in range(f.n_prims))


SCENES = ["p5_linear", "p5_rgrid", "p5_fgrid", "p5_kd", "p5_sah", "p5_convex", "p5_convexsimple", "p2", "p3_run", "p3_mesh",
          "torus100k", "overlap"]


def _scene(name):
    """(flat scene, keep-alive, camera or None, triangles to aim rays at)"""
    if name.startswith("p5_"):
        alg = name[3:]
        s = PresetScene(5, alg, 12 if alg == "linear" else 40)
        return s.flat, s, s.camera, s.triangles()[0]
    if name == "p2":
        s = PresetScene(2)
        return s.flat, s, s.camera, None
    if name.startswith("p3_"):
        s = _preset3(name == "p3_mesh")
        return s.flat, s, s.camera, _loose_tris(s.flat)
    if name == "torus100k":
        tris = _tris_from_facets(rtb200.torus_triangles(100_000, seed=5))
        f = _flat(tris, True)
        return f, f, None, tris
    tris = _ball()
    layout = _overlap_layout(len(tris))
    f = _flat_records(tris, [(rtb200.PRIM_TRIANGLES, 0, 300)] + [(rtb200.PRIM_MESH, a, c) for a, c in layout[1:]])
    return f, f, None, tris


def _rays(cam, tris, seed, n=512):
    rng = np.random.default_rng(seed)
    parts = []
    if cam is not None:
        parts.append(_camera_rays(cam, 64, 48))
    if tris is not None and len(tris):
        parts += list(_ray_sets(tris[rng.permutation(len(tris))[:20000]], rng, n).values())
    if cam is not None:  # random rays from around the eye
        o = np.array(cam.eye, np.float32) + rng.normal(size=(n, 3)).astype(np.float32)
        d = rng.normal(size=(n, 3))
        parts.append(np.concatenate([o, d / np.linalg.norm(d, axis=1, keepdims=True)], 1).astype(np.float32))
    return np.ascontiguousarray(np.concatenate(parts), np.float32)


def _bounds(t, rng):
    """Per-ray bounds around the unbounded distance t (-1 = miss): exactly t, its neighbours, t / 2, 2 t, the special values,
    and uniform draws in between."""
    n = len(t)
    hit = t > 0
    tt = np.where(hit, t, np.float32(rng.uniform(1, 3000))).astype(np.float32)
    kind = rng.integers(0, 13, n)
    b = np.empty(n, np.float32)
    table = [tt, np.nextafter(tt, np.float32(np.inf)), np.nextafter(tt, np.float32(-np.inf)), tt / 2, tt * 2,
             np.full(n, 0.0005, np.float32), np.zeros(n, np.float32), np.full(n, -1, np.float32), np.full(n, np.nan, np.float32),
             np.full(n, np.inf, np.float32), np.full(n, FLT_MAX, np.float32), (rng.uniform(0, 2, n) * tt).astype(np.float32),
             rng.uniform(0.0005, 5000, n).astype(np.float32)]
    for k, v in enumerate(table):
        b[kind == k] = v[kind == k]
    return b


def _masked(res, bound):
    """rtb_intersect_rays results with every hit at t >= bound (or NaN bound) turned into a miss."""
    hid, ht, pos, nrm = (x.copy() for x in res)
    keep = (hid >= 0) & (ht < bound)
    hid[~keep], ht[~keep] = -1, -1
    pos[~keep], nrm[~keep] = 0, 0
    return hid, ht, pos, nrm


def _same(a, b):
    """per-ray bitwise equality of two closest results"""
    eq = (a[0] == b[0]) & (a[1].view(np.uint32) == b[1].view(np.uint32))
    return eq & np.all(a[2].view(np.uint32) == b[2].view(np.uint32), 1) & np.all(a[3].view(np.uint32) == b[3].view(np.uint32), 1)


def _mesh_tri(flat, hit_id):
    """loose record of hit id `hit_id` if a MESH record owns it, else None"""
    f = flat.contents if hasattr(flat, "contents") else flat
    for i in range(f.n_prims):
        p = f.prims[i]
        if p.type == rtb200.PRIM_MESH and p.base_id <= hit_id < p.base_id + p.count:
            return np.ctypeslib.as_array(f.loose_tri, shape=(f.n_loose, 12))[p.first + hit_id - p.base_id]
    return None


def _band_check(flat, rays, run_ids, diff, what):
    """every ray in `diff` must have its run winner in a mesh record and in the grazing band"""
    for i in np.nonzero(diff)[0]:
        tri = _mesh_tri(flat, int(run_ids[i]))
        assert tri is not None and _in_grazing_band(tri, rays[i]), f"{what}: ray {i} differs outside the grazing band"
    print(f"{what}: {len(rays)} rays, {int(diff.sum())} differ in the grazing band")


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


def _np(res):
    return tuple(x.cpu().numpy() for x in res)


# ---- 1-3: results -------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", SCENES)
def test_query_results(ctx, name):
    """Unbounded closest == rtb_intersect_rays bit for bit; bounded closest == the run's unbounded result masked by the bound
    (bit-exact without meshes); ANY == (bounded closest hits)."""
    import torch
    flat, keep, cam, tris = _scene(name)
    mesh = _has_mesh(flat)
    s = ctx.upload(flat)
    run = ctx.upload(_run_twin(flat)) if mesh else s
    try:
        rays = _rays(cam, tris, 41)
        ref = s.intersect_rays(rays)
        rt = _t(rays)
        got = _np(s.query(rt))
        assert _same(got, ref).all(), f"{name}: unbounded query differs from rtb_intersect_rays"
        assert _same(_np(s.query(rt, tmax=float("inf"))), ref).all()
        run_ref = run.intersect_rays(rays) if mesh else ref
        rng = np.random.default_rng(42)
        for rep in range(2):
            bound = _bounds(run_ref[1], rng)
            exp = _masked(run_ref, bound)
            got = _np(s.query(rt, tmax=_t(bound)))
            diff = ~_same(got, exp)
            if mesh:
                _band_check(flat, rays, exp[0], diff, f"{name} bounded")
            else:
                assert not diff.any(), f"{name}: bounded query differs on {int(diff.sum())} rays"
            occ = s.query(rt, tmax=_t(bound), any_hit=True).cpu().numpy()
            assert occ.dtype == np.bool_
            odiff = occ != (exp[0] >= 0)
            if mesh:
                _band_check(flat, rays, exp[0], odiff, f"{name} any")
            else:
                assert not odiff.any(), f"{name}: occlusion differs from the bounded closest hit on {int(odiff.sum())} rays"
            occ_self = s.query(rt, tmax=_t(bound), any_hit=True).cpu().numpy()
            assert np.array_equal(occ, occ_self)
        # one bound for every ray
        for b in (0.0005, 0.0, float("nan"), 50.0, float(FLT_MAX)):
            exp = _masked(run_ref, np.float32(b))
            got = _np(s.query(rt, tmax=b))
            occ = s.query(rt, tmax=b, any_hit=True).cpu().numpy()
            if mesh:
                _band_check(flat, rays, exp[0], ~_same(got, exp), f"{name} tmax={b}")
                _band_check(flat, rays, exp[0], occ != (exp[0] >= 0), f"{name} any tmax={b}")
            else:
                assert _same(got, exp).all() and np.array_equal(occ, exp[0] >= 0), f"{name}: tmax={b}"
        torch.cuda.synchronize()
    finally:
        s.close()
        if run is not s:
            run.close()
        del keep


def _shadow_rays(tris, rng, n, light):
    """rays from surface points (a little off the surface) to a point light, with tmax = distance to the light"""
    v = tris[:, :9].reshape(-1, 3, 3).astype(np.float64)
    k = rng.integers(0, len(tris), n)
    p = np.einsum("ni,nij->nj", rng.dirichlet([1, 1, 1], n), v[k])
    d = light[None, :] - p
    dist = np.linalg.norm(d, axis=1)
    d /= dist[:, None]
    return np.concatenate([p, d], 1).astype(np.float32), dist.astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["p5_sah", "p5_rgrid", "p3_run", "p3_mesh", "torus100k"])
def test_shadow_rays(ctx, name):
    flat, keep, cam, tris = _scene(name)
    mesh = _has_mesh(flat)
    s = ctx.upload(flat)
    run = ctx.upload(_run_twin(flat)) if mesh else s
    try:
        v = tris[:, :9].reshape(-1, 3)
        lo, hi = v.min(0), v.max(0)
        light = (hi + np.array([0.3, 0.5, 0.2]) * (hi - lo)).astype(np.float64)  # outside the model: its far side is in shadow
        rays, dist = _shadow_rays(tris, np.random.default_rng(43), 20000, light)
        exp = _masked(run.intersect_rays(rays), dist)
        occ = s.query(_t(rays), tmax=_t(dist), any_hit=True).cpu().numpy()
        got = _np(s.query(_t(rays), tmax=_t(dist)))
        print(f"{name}: {int(occ.sum())} of {len(rays)} shadow rays occluded")
        if mesh:
            _band_check(flat, rays, exp[0], occ != (exp[0] >= 0), f"{name} shadow any")
            _band_check(flat, rays, exp[0], ~_same(got, exp), f"{name} shadow closest")
        else:
            assert np.array_equal(occ, exp[0] >= 0) and _same(got, exp).all()
    finally:
        s.close()
        if run is not s:
            run.close()
        del keep


@pytest.mark.gpu
def test_torus_1m_any_equals_bounded_closest(ctx):
    tris = _tris_from_facets(rtb200.torus_triangles(1_000_000, seed=6))
    f = _flat(tris, True)
    s = ctx.upload(f)
    try:
        rng = np.random.default_rng(44)
        rays = np.concatenate(list(_ray_sets(tris, rng, 8192).values()))
        closest = _np(s.query(_t(rays)))
        bound = _bounds(closest[1], rng)
        bc = _np(s.query(_t(rays), tmax=_t(bound)))
        occ = s.query(_t(rays), tmax=_t(bound), any_hit=True).cpu().numpy()
        _band_check(f, rays, bc[0], occ != (bc[0] >= 0), "1M any vs bounded closest")
    finally:
        s.close()


# ---- 4: streams ---------------------------------------------------------------------------------
def _mesh_scene(ctx, n=1_000_000):
    tris = _tris_from_facets(rtb200.torus_triangles(n, seed=6))
    return tris, ctx.upload(_flat(tris, True, lead_sphere=False))


def _torch_rays(tris, n, seed):
    """camera-like rays made by torch ops on the current stream: points on a sphere around the model, aimed into its box"""
    import torch
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    v = torch.from_numpy(tris[:, :9].reshape(-1, 3)).to("cuda:0")
    lo, hi = v.min(0).values, v.max(0).values
    c, ext = (lo + hi) / 2, float((hi - lo).max())
    o = torch.randn(n, 3, device="cuda:0", generator=g)
    o = c + o / o.norm(dim=1, keepdim=True) * ext * 1.5
    tgt = lo + torch.rand(n, 3, device="cuda:0", generator=g) * (hi - lo)
    d = tgt - o
    return torch.cat([o, d / d.norm(dim=1, keepdim=True)], 1).contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["side", "default"])
def test_rays_from_torch_on_a_stream(ctx, where):
    """Rays and bounds produced by torch on a stream, queried there with no synchronise and overwritten right after the call:
    the query reads them after the producing ops and before the overwrite."""
    import torch
    tris, s = _mesh_scene(ctx)
    try:
        torch.cuda.synchronize()
        st = torch.cuda.Stream(device=0) if where == "side" else torch.cuda.default_stream(0)
        with torch.cuda.stream(st):
            rays = _torch_rays(tris, 1 << 20, 7)
            for _ in range(4):  # enough work ahead of the query that a missing wait would read unfinished rays
                rays = torch.cat([rays[:, :3], rays[:, 3:] / rays[:, 3:].norm(dim=1, keepdim=True)], 1).contiguous()
            tmax = (rays[:, 0].abs() + 20.0).contiguous()
            expected_rays, expected_tmax = rays.clone(), tmax.clone()
            got = s.query(rays, tmax=tmax)
            occ = s.query(rays, tmax=tmax, any_hit=True)
            rays.fill_(float("nan"))
            tmax.fill_(0.0)
        torch.cuda.synchronize()
        r, b = expected_rays.cpu().numpy(), expected_tmax.cpu().numpy()
        exp = _masked(s.intersect_rays(r), b)
        assert _same(_np(got), exp).all()
        assert np.array_equal(occ.cpu().numpy(), exp[0] >= 0)
    finally:
        s.close()


@pytest.mark.gpu
def test_query_does_not_synchronise(ctx):
    """A query queued behind a long sleep returns while its stream is still busy."""
    import torch
    tris, s = _mesh_scene(ctx, 100_000)
    try:
        rays = _torch_rays(tris, 4096, 8)
        torch.cuda.synchronize()
        st = torch.cuda.Stream(device=0)
        with torch.cuda.stream(st):
            torch.cuda._sleep(1_000_000_000)  # about half a second
            got = s.query(rays)
            occ = s.query(rays, tmax=10.0, any_hit=True)
        busy = not st.query()
        st.synchronize()
        assert busy, "the query call waited for its stream"
        r = rays.cpu().numpy()
        assert _same(_np(got), s.intersect_rays(r)).all()
        assert np.array_equal(occ.cpu().numpy(), _masked(s.intersect_rays(r), np.float32(10.0))[0] >= 0)
    finally:
        s.close()


# ---- 5: ordering against updates and renders ----------------------------------------------------
@pytest.mark.gpu
def test_query_is_ordered_before_a_later_update(ctx):
    """A large query on stream A, then an update of the mesh on stream B: the query sees the old triangles; a query after the
    update sees the new ones."""
    import torch
    tris, s = _mesh_scene(ctx)
    new = twist(tris, 0.6, 1.05)
    old_ref = ctx.upload(_flat(tris, True, lead_sphere=False))
    new_ref = ctx.upload(_flat(new, True, lead_sphere=False))
    try:
        rays = _torch_rays(tris, 1 << 22, 9)
        rec = _t(new)
        torch.cuda.synchronize()
        sa, sb = torch.cuda.Stream(device=0), torch.cuda.Stream(device=0)
        with torch.cuda.stream(sa):
            torch.cuda._sleep(200_000_000)  # the query is still queued when the update is enqueued
            before = s.query(rays)
            before_occ = s.query(rays, tmax=25.0, any_hit=True)
        with torch.cuda.stream(sb):
            s.mesh_update(rec)
        with torch.cuda.stream(sa):
            after = s.query(rays)
        torch.cuda.synchronize()
        for got, ref, what in ((before, old_ref, "before"), (after, new_ref, "after")):
            assert all(torch.equal(g, e) for g, e in zip(got, ref.query(rays))), f"the query {what} the update"
        assert torch.equal(before_occ, old_ref.query(rays, tmax=25.0, any_hit=True))
        assert not torch.equal(before[0], after[0])
        sub = slice(0, 1 << 16)
        assert _same(tuple(x[sub].cpu().numpy() for x in before), old_ref.intersect_rays(rays[sub].cpu().numpy())).all()
    finally:
        s.close()
        old_ref.close()
        new_ref.close()


@pytest.mark.gpu
def test_render_and_query_on_other_streams_precede_an_update(ctx):
    import torch
    ball = _ball()
    new = twist(ball, 0.8, 1.1)
    a = _preset3(True)
    frame = rtb200.make_frame(400, 300, samples=4, seed=7)
    d = ctx.upload(a.flat)
    try:
        ref_img = torch.zeros((300, 400, 3), dtype=torch.float32, device="cuda:0")
        d.render_device(a.camera, a.setting, frame, ref_img.data_ptr())
        rays = _t(_rays(a.camera, ball, 45))
        ref_q = d.query(rays)
        torch.cuda.synchronize()
        s1, s2, s3 = (torch.cuda.Stream(device=0) for _ in range(3))
        out = torch.zeros((300, 400, 3), dtype=torch.float32, device="cuda:0")
        with torch.cuda.stream(s1):
            torch.cuda._sleep(200_000_000)
        d.render_device(a.camera, a.setting, frame, out.data_ptr(), stream=s1.cuda_stream)
        with torch.cuda.stream(s2):
            torch.cuda._sleep(200_000_000)
            q = d.query(rays)
        with torch.cuda.stream(s3):
            d.mesh_update(_t(new))
            after = d.query(rays)
        torch.cuda.synchronize()
        assert torch.equal(out, ref_img), "the render before the update saw the new triangles"
        assert all(torch.equal(x, y) for x, y in zip(q, ref_q)), "the query before the update saw the new triangles"
        assert not torch.equal(after[0], ref_q[0]), "the query after the update did not see the new triangles"
    finally:
        d.close()
        a.close()


# ---- 6: refusals --------------------------------------------------------------------------------
def _raw(ctx, scene, n, rays, tmax, flags, hid=None, ht=None, pos=None, nrm=None, occ=None, stream=None):
    p = lambda x: None if x is None else C.c_void_p(x if isinstance(x, int) else x.data_ptr())
    return ctx._lib.rtb_query_rays(ctx._h, scene._h, n, p(rays), p(tmax), float("inf"), flags, p(hid), p(ht), p(pos), p(nrm),
                                   p(occ), p(stream))


@pytest.mark.gpu
def test_refused_calls_write_nothing(ctx):
    import torch
    tris = _ball()
    s = ctx.upload(_flat(tris, True))
    try:
        rays_np = _rays(None, tris, 46, 256)
        n = len(rays_np)
        rays = _t(rays_np)
        tmax = torch.full((n,), 100.0, device="cuda:0")
        hid = torch.full((n,), 12345, dtype=torch.int32, device="cuda:0")
        ht = torch.full((n,), 7.5, device="cuda:0")
        pos = torch.full((n, 3), 7.5, device="cuda:0")
        nrm = torch.full((n, 3), 7.5, device="cuda:0")
        occ = torch.full((n,), 77, dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()
        snap = [x.clone() for x in (hid, ht, pos, nrm, occ)]
        CL, ANY = rtb200.QUERY_CLOSEST, rtb200.QUERY_ANY
        host = np.ascontiguousarray(rays_np)
        pinned = rtb200.PinnedArray((n, 6))
        pinned.array[:] = rays_np
        mis = torch.zeros(n * 6 + 1, device="cuda:0")
        mis[1:] = rays.view(-1)
        torch.cuda.synchronize()
        cases = {
            "host rays": _raw(ctx, s, n, host.ctypes.data, None, CL, hid, ht, pos, nrm),
            "page-locked host rays": _raw(ctx, s, n, pinned._p.value, None, CL, hid, ht, pos, nrm),
            "host tmax": _raw(ctx, s, n, rays, np.full(n, 5, np.float32).ctypes.data, CL, hid, ht, pos, nrm),
            "misaligned rays": _raw(ctx, s, n, mis[1:].data_ptr(), None, CL, hid, ht, pos, nrm),
            "n < 0": _raw(ctx, s, -1, rays, None, CL, hid, ht, pos, nrm),
            "unknown flags": _raw(ctx, s, n, rays, None, 2, hid, ht, pos, nrm),
            "ANY with closest outputs": _raw(ctx, s, n, rays, tmax, ANY, hid, occ=occ),
            "ANY without occluded": _raw(ctx, s, n, rays, tmax, ANY),
            "CLOSEST with occluded": _raw(ctx, s, n, rays, tmax, CL, hid, ht, pos, nrm, occ),
            "misaligned output": _raw(ctx, s, n, rays, tmax, CL, ht.data_ptr() + 2),
        }
        torch.cuda.synchronize()
        pinned.close()
        for what, rc in cases.items():
            assert rc == ERR_INVALID, f"{what}: rc {rc}"
        for a, b in zip((hid, ht, pos, nrm, occ), snap):
            assert torch.equal(a, b), "a refused call wrote its outputs"
        assert _raw(ctx, s, 0, None, None, CL) == 0  # n == 0: nothing to do
        with pytest.raises(rtb200.RtbError):
            s.query(rays.cpu())
        with pytest.raises(rtb200.RtbError):
            s.query(rays, tmax=tmax[:-1])
    finally:
        s.close()


# ---- 7: constants (no device) -------------------------------------------------------------------
def test_header_query_flags_match_the_bindings():
    text = open(os.path.join(rtb200.ROOT, "include", "rtb.h")).read()
    assert re.search(r"enum \{ RTB_QUERY_CLOSEST = 0, RTB_QUERY_ANY = 1 \};", text)
    assert (rtb200.QUERY_CLOSEST, rtb200.QUERY_ANY) == (0, 1)
    assert "rtb_query_rays" in rtb200.ABI_SYMBOLS
