"""RTB_PRIM_MESH: a triangle mesh traversed through a hierarchy built on the device must return, ray for ray, what the run of
loose triangles with the same records returns (include/rtb.h), except where the run's winning pair lies in the grazing band
of csrc/rtb_bvh.h.  The run is the oracle, on the GPU itself."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import rtb200
from rtb200 import PresetScene

HEADER = os.path.join(rtb200.ROOT, "include", "rtb.h")
BVH_H = os.path.join(rtb200.PKG, "csrc", "rtb_bvh.h")


def _preset3(mesh, stl=None):
    rtb200.set_stl_as_mesh(mesh)
    try:
        return PresetScene(3, stl_path=stl)
    finally:
        rtb200.set_stl_as_mesh(False)


def _prims(flat):
    f = flat.contents
    return [(p.type, p.material, p.base_id, p.first, p.count) for p in f.prims[:f.n_prims]]


def _loose(flat):
    f = flat.contents
    return np.ctypeslib.as_array(f.loose_tri, shape=(f.n_loose * 12,)).copy()


# ---- host side (no device) --------------------------------------------------------------------
def test_header_constants_match_the_documented_enum():
    text = open(HEADER).read()
    assert re.search(r"RTB_PRIM_MESH = 4", text)
    assert re.search(r"#define RTB_ABI_VERSION 5\b", text)
    assert (rtb200.PRIM_PLANE, rtb200.PRIM_SPHERE, rtb200.PRIM_TRIANGLES, rtb200.PRIM_TUNNEL, rtb200.PRIM_MESH) == (0, 1, 2, 3, 4)
    assert C.sizeof(rtb200.BvhNode) == 64
    assert "rtb_scene_mesh_download" in rtb200.ABI_SYMBOLS
    bvh = open(BVH_H).read()
    assert "#define RTB_BVH_C 1024.0f" in bvh and "#define RTB_BVH_STACK 64" in bvh
    # the widening factor covers 1 / C and the roundings the header lists
    k = float(re.search(r"#define RTB_BVH_K ([0-9.e-]+)f", bvh).group(1))
    u = 2.0 ** -24
    assert k >= (1 / 1024 + u) * (1 + u) * (1 + 4 * u)


def test_stl_mesh_flattens_to_the_same_records_as_the_run():
    run, mesh = _preset3(False), _preset3(True)
    try:
        fr, fm = run.flat.contents, mesh.flat.contents
        assert fm.n_top == fr.n_top and fm.n_loose == fr.n_loose == 528
        assert np.array_equal(_loose(run.flat), _loose(mesh.flat))
        pr, pm = _prims(run.flat), _prims(mesh.flat)
        runs = [p for p in pr if p[0] == rtb200.PRIM_TRIANGLES]
        meshes = [p for p in pm if p[0] == rtb200.PRIM_MESH]
        assert len(runs) == 1 and len(meshes) == 1
        assert meshes[0][1:] == runs[0][1:]  # material, base_id, first, count
        assert [p for p in pm if p[0] != rtb200.PRIM_MESH] == [p for p in pr if p[0] != rtb200.PRIM_TRIANGLES]
        assert pm.index(meshes[0]) == pr.index(runs[0])
        mats_r = bytes(C.string_at(C.addressof(fr.materials.contents), 64 * fr.n_materials))
        mats_m = bytes(C.string_at(C.addressof(fm.materials.contents), 64 * fm.n_materials))
        assert mats_r == mats_m
    finally:
        run.close()
        mesh.close()


def test_torus_stl_round_trip(tmp_path):
    facets = rtb200.torus_triangles(2000, seed=3)
    path = str(tmp_path / "torus.stl")
    rtb200.write_stl(path, facets)
    run, mesh = _preset3(False, path), _preset3(True, path)
    try:
        assert run.flat.contents.n_loose == mesh.flat.contents.n_loose == len(facets)
        assert np.array_equal(_loose(run.flat), _loose(mesh.flat))
        assert [p[0] for p in _prims(mesh.flat)].count(rtb200.PRIM_MESH) == 1
    finally:
        run.close()
        mesh.close()


def test_node_test_bound_on_the_cpu(tmp_path):
    """csrc/rtb_bvh.h compiled for the host: for 200 k random pairs the reference's test accepts outside the grazing band
    (random, nearly grazing, zero and denormal direction components, aim points on the edge of the -1e-4 slack), the node
    test visits the triangle's leaf box and an enclosing box with best = the accepted t."""
    exe = str(tmp_path / "bvh_bound_check")
    src = os.path.join(rtb200.ROOT, "tests", "bvh_bound_check.cpp")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-o", exe, src])
    for seed in (1, 2):
        out = subprocess.run([exe, str(seed), "200000"], capture_output=True, text=True)
        print(out.stdout)
        assert out.returncode == 0, out.stdout
        counts = dict(re.findall(r"(\w+) (\d+)", out.stdout.splitlines()[-1]))
        assert int(counts["violations"]) == 0 and int(counts["checked"]) == 200000
        assert int(counts["zero_dir"]) > 1000 and int(counts["denormal_dir"]) > 1000 and int(counts["grazing"]) > 1000


# ---- CPU model of the reference's determinant and of the grazing band (csrc/rtb_bvh.h) ----------
def _det3_ref(a11, a12, a13, a21, a22, a23, a31, a32, a33):
    f = np.float32
    return f(f(f(f(f(f(a11 * a22) * a33) + f(f(a12 * a23) * a31)) + f(f(a13 * a21) * a32)) - f(f(a13 * a22) * a31))
             - f(f(a11 * a23) * a32)) - f(f(a12 * a21) * a33)


def _in_grazing_band(tri, ray):
    """tri: 12 floats a, b, c, n; ray: 6 floats.  |detM_r| <= C kappa_g, kappa_g = 2^-19 dmx (A1 + E^2)."""
    f = np.float32
    t = np.asarray(tri, np.float32)
    d = np.asarray(ray[3:6], np.float32)
    e1 = np.array([f(t[0] - t[3]), f(t[1] - t[4]), f(t[2] - t[5])], np.float32)
    e2 = np.array([f(t[0] - t[6]), f(t[1] - t[7]), f(t[2] - t[8])], np.float32)
    det = _det3_ref(e1[0], e2[0], d[0], e1[1], e2[1], d[1], e1[2], e2[2], d[2])
    x1, y1, z1 = np.abs(e1.astype(np.float64))
    x2, y2, z2 = np.abs(e2.astype(np.float64))
    a1 = x1 * (y2 + z2) + y1 * (x2 + z2) + z1 * (x2 + y2)
    e = max(x1 + y1 + z1, x2 + y2 + z2)
    kappa = 2.0 ** -19 * float(np.max(np.abs(d))) * (a1 + e * e)
    return abs(float(det)) <= 1024.0 * kappa


# ---- device side ------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    c = rtb200.Context(0)
    yield c
    c.close()


def _flat(tris, mesh, lead_sphere=True):
    """A flat scene of one sphere (a record before the triangles) and the triangles as a run or a mesh."""
    tris = np.ascontiguousarray(tris, np.float32).reshape(-1, 12)
    n = len(tris)
    mats = (rtb200.Material * 1)()
    mats[0].kind, mats[0].diffusiveness = 0, 1.0
    mats[0].a[0] = mats[0].a[1] = mats[0].a[2] = 0.5
    prims = (rtb200.Prim * 2)()
    k = 0
    if lead_sphere:
        c = tris[:, :9].reshape(-1, 3).mean(0)
        prims[0].type, prims[0].base_id = rtb200.PRIM_SPHERE, 0
        prims[0].v[0], prims[0].v[1], prims[0].v[2], prims[0].v[3] = float(c[0]) + 1000.0, float(c[1]), float(c[2]), 1.0
        k = 1
    p = prims[k]
    p.type, p.material, p.base_id, p.first, p.count = (rtb200.PRIM_MESH if mesh else rtb200.PRIM_TRIANGLES), 0, k, 0, n
    f = rtb200.FlatScene()
    f.n_prims, f.prims, f.n_materials, f.materials = k + 1, prims, 1, mats
    f.n_top, f.n_loose = k + n, n
    f.loose_tri = tris.ctypes.data_as(C.POINTER(C.c_float))
    f._keep = (tris, mats, prims)
    return f


def _compare(ctx, tris, rays, what, lead_sphere=True):
    """Run vs mesh through rtb_intersect_rays: bit-identical except on rays whose run winner lies in the grazing band
    (checked here on the CPU).  Returns the number of such rays."""
    tris = np.ascontiguousarray(tris, np.float32).reshape(-1, 12)
    rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 6)
    fr, fm = _flat(tris, False, lead_sphere), _flat(tris, True, lead_sphere)
    sr, sm = ctx.upload(fr), ctx.upload(fm)
    try:
        r = sr.intersect_rays(rays)
        m = sm.intersect_rays(rays)
    finally:
        sr.close()
        sm.close()
    base = 1 if lead_sphere else 0
    same = (r[0] == m[0]) & (r[1].view(np.uint32) == m[1].view(np.uint32)) & \
        np.all(r[2].view(np.uint32) == m[2].view(np.uint32), 1) & np.all(r[3].view(np.uint32) == m[3].view(np.uint32), 1)
    band = 0
    for i in np.nonzero(~same)[0]:
        k = int(r[0][i]) - base
        assert 0 <= k < len(tris), f"{what}: ray {i}: run {r[0][i]} {r[1][i]} vs mesh {m[0][i]} {m[1][i]}"
        assert _in_grazing_band(tris[k], rays[i]), f"{what}: ray {i} differs outside the grazing band: run {r[0][i]} {r[1][i]} " \
                                                   f"vs mesh {m[0][i]} {m[1][i]}"
        band += 1
    print(f"{what}: {len(rays)} rays, {int(np.sum(r[0] >= base))} hits, {band} differ in the grazing band")
    return band


def _tris_from_facets(facets, offset=(0.0, 0.0, 0.0)):
    f = np.asarray(facets, np.float32)
    o = np.asarray(offset, np.float32)
    v = f[:, 3:12].reshape(-1, 3, 3) + o
    return np.concatenate([v.reshape(-1, 9), f[:, :3]], 1).astype(np.float32)


def _ball():
    s = PresetScene(3)
    try:
        return _loose(s.flat).reshape(-1, 12)
    finally:
        s.close()


def _norm(d):
    return (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)


def _ray_sets(tris, rng, n):
    v = tris[:, :9].reshape(-1, 3, 3).astype(np.float64)
    lo, hi = v.reshape(-1, 3).min(0), v.reshape(-1, 3).max(0)
    c, ext = (lo + hi) / 2, float(np.max(hi - lo))
    sets = {}
    # camera-like rays: from points on a sphere around the model towards random points of its box
    o = c + _norm(rng.normal(size=(n, 3))) * ext * 1.5
    tgt = lo + rng.uniform(size=(n, 3)) * (hi - lo)
    sets["camera"] = np.concatenate([o, _norm(tgt - o)], 1)
    # from surface points (barycentric interior) in random and nearly tangent directions
    k = rng.integers(0, len(tris), n)
    w = rng.dirichlet([1, 1, 1], n)
    p = np.einsum("ni,nij->nj", w, v[k])
    nrm = np.cross(v[k, 1] - v[k, 0], v[k, 2] - v[k, 0])
    nrm = nrm / np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-30)
    d = _norm(rng.normal(size=(n, 3)))
    sets["surface_random"] = np.concatenate([p, d], 1)
    tang = d - nrm * np.sum(d * nrm, 1, keepdims=True)
    tang = _norm(tang + nrm * rng.uniform(-1e-3, 1e-3, (n, 1)))
    sets["surface_tangent"] = np.concatenate([p, tang], 1)
    # through vertices and along edges
    vert = v[k, rng.integers(0, 3, n)]
    sets["vertices"] = np.concatenate([o, _norm(vert - o)], 1)
    a, b = v[k, 0], v[k, 1]
    sets["edges"] = np.concatenate([a - (b - a) * 2.0, _norm(b - a)], 1)
    # axis-parallel rays (two zero direction components)
    ax = rng.integers(0, 3, n)
    dd = np.zeros((n, 3))
    dd[np.arange(n), ax] = rng.choice([-1.0, 1.0], n)
    oo = lo + rng.uniform(size=(n, 3)) * (hi - lo)
    oo[np.arange(n), ax] = np.where(dd[np.arange(n), ax] > 0, lo[ax] - ext, hi[ax] + ext)
    sets["axis_parallel"] = np.concatenate([oo, dd], 1)
    return {name: r.astype(np.float32) for name, r in sets.items()}


@pytest.mark.gpu
def test_mesh_equals_run_ball(ctx):
    tris = _ball()
    band = sum(_compare(ctx, tris, rays, "ball " + name) for name, rays in _ray_sets(tris, np.random.default_rng(1), 4096).items())
    print("ball: grazing-band rays", band)


@pytest.mark.gpu
def test_mesh_equals_run_100k(ctx):
    tris = _tris_from_facets(rtb200.torus_triangles(100_000, seed=5))
    band = sum(_compare(ctx, tris, rays, "100k " + name) for name, rays in _ray_sets(tris, np.random.default_rng(2), 2048).items())
    print("100k: grazing-band rays", band)


@pytest.mark.gpu
def test_mesh_equals_run_1m_sample(ctx):
    tris = _tris_from_facets(rtb200.torus_triangles(1_000_000, seed=6))
    sets = _ray_sets(tris, np.random.default_rng(3), 683)
    rays = np.concatenate(list(sets.values()))[:4096]
    print("1M: grazing-band rays", _compare(ctx, tris, rays, "1M sample"))


@pytest.mark.gpu
def test_mesh_equals_run_special_meshes(ctx):
    rng = np.random.default_rng(4)
    ball = _ball()
    # duplicated triangles: the tie must go to the lowest index
    dup = np.concatenate([ball, ball[::-1], ball])
    # zero-area facets mixed in (a collapsed vertex, three equal vertices)
    zero = ball.copy()
    zero[::7, 3:6] = zero[::7, 0:3]
    zero[3::11, 3:9] = np.tile(zero[3::11, 0:3], 2)
    # a coplanar tessellated plate (z = 0)
    g = np.linspace(-10, 10, 41, dtype=np.float32)
    x, y = np.meshgrid(g, g, indexing="ij")
    q = np.stack([x, y, np.zeros_like(x)], -1)
    a, b, c, d = q[:-1, :-1], q[1:, :-1], q[1:, 1:], q[:-1, 1:]
    plate_v = np.concatenate([np.stack([a, b, c], -2).reshape(-1, 9), np.stack([a, c, d], -2).reshape(-1, 9)])
    plate = np.concatenate([plate_v, np.tile([0, 0, 1], (len(plate_v), 1))], 1).astype(np.float32)
    # the ball moved by 1e4
    far = ball.copy()
    far[:, :9] += np.float32(1e4)
    # every centroid at the same point: triangles rotated about a common centre
    ang = rng.uniform(0, 2 * np.pi, (500, 3))
    base_t = np.array([[1, 0, 0], [-0.5, 0.8, 0], [-0.5, -0.8, 0]], np.float64)
    cen = []
    for a0, a1, a2 in ang:
        rz = np.array([[np.cos(a0), -np.sin(a0), 0], [np.sin(a0), np.cos(a0), 0], [0, 0, 1]])
        rx = np.array([[1, 0, 0], [0, np.cos(a1), -np.sin(a1)], [0, np.sin(a1), np.cos(a1)]])
        t = base_t @ (rx @ rz).T * (1 + a2)
        t -= t.mean(0)
        cen.append(np.concatenate([t.reshape(9), [0, 0, 1]]))
    cen = np.asarray(cen, np.float32)
    total = 0
    for name, tris in [("duplicates", dup), ("zero_area", zero), ("plate", plate), ("offset_1e4", far), ("same_centroid", cen)]:
        for rname, rays in _ray_sets(tris, rng, 2048).items():
            total += _compare(ctx, tris, rays, f"{name} {rname}")
    print("special meshes: grazing-band rays", total)


def _flat_records(tris, records):
    """records: [(type, first, count)] over one loose array; record j has base_id = first (ids are the loose indices)."""
    tris = np.ascontiguousarray(tris, np.float32).reshape(-1, 12)
    mats = (rtb200.Material * 1)()
    mats[0].kind, mats[0].diffusiveness = 0, 1.0
    prims = (rtb200.Prim * len(records))()
    for j, (typ, first, count) in enumerate(records):
        prims[j].type, prims[j].material, prims[j].base_id, prims[j].first, prims[j].count = typ, 0, first, first, count
    f = rtb200.FlatScene()
    f.n_prims, f.prims, f.n_materials, f.materials = len(records), prims, 1, mats
    f.n_top, f.n_loose = len(tris), len(tris)
    f.loose_tri = tris.ctypes.data_as(C.POINTER(C.c_float))
    f._keep = (tris, mats, prims)
    return f


@pytest.mark.gpu
def test_overlapping_mesh_records_each_get_their_own_tree(ctx):
    """Mesh records whose loose ranges overlap (and a run in front of them) hit what runs over the same ranges hit."""
    tris = _ball()
    n = len(tris)
    layout = [(0, 300), (200, n - 200), (100, 150), (0, n)]
    run = _flat_records(tris, [(rtb200.PRIM_TRIANGLES, a, c) for a, c in layout])
    mesh = _flat_records(tris, [(rtb200.PRIM_TRIANGLES, 0, 300)] + [(rtb200.PRIM_MESH, a, c) for a, c in layout[1:]])
    rays = np.concatenate(list(_ray_sets(tris, np.random.default_rng(11), 2048).values()))
    sr, sm = ctx.upload(run), ctx.upload(mesh)
    try:
        r, m = sr.intersect_rays(rays), sm.intersect_rays(rays)
        dev = sm.device_bytes - sr.device_bytes
        for j in range(3):
            _, _, child, order, depth = sm.mesh_download(j)
            assert sorted(order.tolist()) == list(range(layout[j + 1][1])) and depth <= 63
    finally:
        sr.close()
        sm.close()
    assert dev == sum(c for _, c in layout[1:]) * (64 + 48 + 4)  # sized by the mesh triangles only
    diff = np.nonzero((r[0] != m[0]) | (r[1].view(np.uint32) != m[1].view(np.uint32)))[0]
    for i in diff:
        assert 0 <= r[0][i] < n and _in_grazing_band(tris[r[0][i]], rays[i]), f"ray {i}: run {r[0][i]} {r[1][i]} mesh {m[0][i]} {m[1][i]}"
    assert np.sum(r[0] >= 0) > len(rays) // 2
    print("overlapping records: grazing-band rays", len(diff))


@pytest.mark.gpu
def test_tree_invariants(ctx):
    for tris in (_ball(), _tris_from_facets(rtb200.torus_triangles(100_000, seed=5)), _ball()[:1]):
        f = _flat(tris, True, lead_sphere=False)
        s1, s2 = ctx.upload(f), ctx.upload(f)
        try:
            lo, hi, child, order, depth = s1.mesh_download()
            again = s2.mesh_download()
            dev_bytes = s1.device_bytes
        finally:
            s1.close()
            s2.close()
        n = len(tris)
        for x, y in zip((lo, hi, child, order), again[:4]):
            assert x.tobytes() == y.tobytes(), "two uploads gave different trees"
        assert depth == again[4] and depth <= 63
        assert sorted(order.tolist()) == list(range(n))  # every triangle exactly once
        assert dev_bytes >= n * (64 + 48 + 4)
        if n == 1:
            assert child.tolist() == [[-1, -1]]
            continue
        assert len(child) == n - 1
        leaves = child[child < 0]
        assert sorted((~leaves).tolist()) == list(range(n))
        inner = child[child >= 0]
        assert sorted(inner.tolist()) == list(range(1, n - 1))
        # child boxes nest in the parent's box (the union the parent stores for it)
        for node in range(n - 1):
            for side in range(2):
                c = child[node, side]
                if c >= 0:
                    assert np.all(lo[c].min(0) >= lo[node, side]) and np.all(hi[c].max(0) <= hi[node, side])
        # each leaf box contains its triangle widened by the barycentric slack
        v = tris[:, :9].reshape(-1, 3, 3)
        for node in range(n - 1):
            for side in range(2):
                c = child[node, side]
                if c < 0:
                    t = v[order[~c]]
                    mn, mx = t.min(0), t.max(0)
                    w = (mx - mn) * np.float32(2.0e-4)
                    assert np.all(lo[node, side] <= mn - w) and np.all(hi[node, side] >= mx + w)


def _material_non_refractive(scene):
    f = scene.flat.contents
    for i in range(f.n_materials):
        m = f.materials[i]
        if m.refractiveness > 0:
            m.diffusiveness, m.reflectiveness, m.refractiveness = 0.3, 0.7, 0.0


def _render_pair(ctx, setting, frame, non_refractive=False):
    out = []
    for mesh in (False, True):
        s = _preset3(mesh)
        if non_refractive:
            _material_non_refractive(s)
        d = ctx.upload(s.flat)
        try:
            img, st = d.render(s.camera, setting if setting is not None else s.setting, frame)
        finally:
            d.close()
            s.close()
        out.append((img, st))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["mc", "simple_tree", "chain"])
def test_preset3_images_mesh_equals_run(ctx, kind):
    setting = {"mc": None, "simple_tree": rtb200.make_setting("simple"), "chain": rtb200.make_setting("simple")}[kind]
    frames = [rtb200.make_frame(400, 300, samples=4, seed=7, counters=1),
              rtb200.make_frame(400, 300, samples=4, seed=7, rank=1, world=3, counters=1),
              rtb200.make_frame(400, 300, samples=4, seed=7, rank=1, world=2, col_block=8, counters=1)]
    if kind == "mc":
        frames.append(rtb200.make_frame(400, 300, samples=4, seed=7, sample_first=1, sample_count=2, counters=1))
    for fr in frames:
        (ri, rs), (mi, ms) = _render_pair(ctx, setting, fr, non_refractive=kind == "chain")
        assert ri.tobytes() == mi.tobytes(), f"{kind}: mesh image differs from the run's"
        assert rs["n_rays"] == ms["n_rays"]
        assert ms["n_tri_tests"] < rs["n_tri_tests"]
        print(kind, "tri tests run", rs["n_tri_tests"], "mesh", ms["n_tri_tests"], "kernel ms", rs["kernel_ms"], ms["kernel_ms"])


@pytest.mark.gpu
def test_bounce_rays_mesh_equals_run(ctx):
    tris = _ball()
    rays = _ray_sets(tris, np.random.default_rng(9), 2048)["camera"]
    lib = ctx._lib
    lib.rtb_bounce_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_float)]
    res = []
    for mesh in (False, True):
        s = ctx.upload(_flat(tris, mesh))
        n = len(rays)
        ok, depth, last, pos = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros((n, 3), np.float32)
        total, ms = C.c_int64(0), C.c_float(0)
        try:
            ctx._check(lib.rtb_bounce_rays(ctx._h, s._h, n, rays.ctypes.data, 16, ok.ctypes.data, depth.ctypes.data, last.ctypes.data,
                                           pos.ctypes.data, C.byref(total), C.byref(ms)), "rtb_bounce_rays")
        finally:
            s.close()
        res.append((ok, depth, last, pos, total.value))
    for x, y in zip(res[0], res[1]):
        assert np.asarray(x).tobytes() == np.asarray(y).tobytes()


@pytest.mark.gpu
def test_multi_render_mesh_equals_run():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two or more GPUs")
    m = rtb200.MultiContext(2)
    try:
        imgs = []
        for mesh in (False, True):
            s = _preset3(mesh)
            d = m.upload(s.flat)
            try:
                img, st = d.render(s.camera, s.setting, rtb200.make_frame(400, 300, samples=4, seed=7))
            finally:
                d.close()
                s.close()
            imgs.append((img, st["n_rays"]))
        assert imgs[0][0].tobytes() == imgs[1][0].tobytes() and imgs[0][1] == imgs[1][1]
    finally:
        m.close()
