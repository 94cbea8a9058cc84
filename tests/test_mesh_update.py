"""rtb_scene_mesh_update: a mesh's triangles replaced in place on the device.  A rebuild must give what a fresh upload of the new
records gives, bit for bit; a refit keeps the tree's shape and must keep the mesh's contract (the run's hits, except in the
grazing band of csrc/rtb_bvh.h).  The fresh upload and the run are the oracles, on the GPU itself."""
import ctypes as C

import numpy as np
import pytest

import rtb200
from test_mesh import _ball, _flat, _flat_records, _in_grazing_band, _loose, _material_non_refractive, _preset3, _ray_sets, \
    _tris_from_facets

ERR_INVALID, ERR_UNSUPPORTED = -1, -4


@pytest.fixture(scope="module")
def ctx():
    c = rtb200.Context(0)
    yield c
    c.close()


def twist(tris, amount, scale=1.0):
    """[n][12] records (a, b, c, normal) twisted about the vertical axis through the model's centre by up to `amount` radians
    (growing with height) and scaled about that centre; normals recomputed.  A smooth deformation, as a skinned or simulated
    model moves."""
    v = tris[:, :9].reshape(-1, 3).astype(np.float64)
    lo, hi = v.min(0), v.max(0)
    c = (lo + hi) / 2
    p = (v - c) * scale
    a = amount * (v[:, 1] - lo[1]) / max(hi[1] - lo[1], 1e-30)
    x = p[:, 0] * np.cos(a) - p[:, 2] * np.sin(a)
    z = p[:, 0] * np.sin(a) + p[:, 2] * np.cos(a)
    w = (np.stack([x, p[:, 1], z], 1) + c).astype(np.float32).reshape(-1, 3, 3)
    n = np.cross(w[:, 1] - w[:, 0], w[:, 2] - w[:, 0])
    n /= np.maximum(np.linalg.norm(n, axis=1, keepdims=True), 1e-30)
    return np.concatenate([w.reshape(-1, 9), n.astype(np.float32)], 1).astype(np.float32)


def _model(name):
    if name == "ball":
        return _ball()
    if name == "torus100k":
        return _tris_from_facets(rtb200.torus_triangles(100_000, seed=5))
    return _ball()[:1]


def _tree_bytes(scene, mesh_index=0):
    lo, hi, child, order, depth = scene.mesh_download(mesh_index)
    return lo.tobytes(), hi.tobytes(), child.tobytes(), order.tobytes(), depth


def _hits(scene, rays):
    return [x.tobytes() for x in scene.intersect_rays(rays)]


def _all_rays(tris, seed, n=1024):
    return np.concatenate(list(_ray_sets(tris, np.random.default_rng(seed), n).values()))


def _band_only(tris, rays, run, mesh, what):
    """run vs mesh intersect_rays results (no record before the mesh): equal except on rays whose run winner lies in the
    grazing band.  Returns the number of such rays."""
    same = (run[0] == mesh[0]) & (run[1].view(np.uint32) == mesh[1].view(np.uint32))
    same &= np.all(run[2].view(np.uint32) == mesh[2].view(np.uint32), 1) & np.all(run[3].view(np.uint32) == mesh[3].view(np.uint32), 1)
    diff = np.nonzero(~same)[0]
    for i in diff:
        k = int(run[0][i])
        assert 0 <= k < len(tris) and _in_grazing_band(tris[k], rays[i]), \
            f"{what}: ray {i} differs outside the grazing band: run {run[0][i]} {run[1][i]} vs mesh {mesh[0][i]} {mesh[1][i]}"
    print(f"{what}: {len(rays)} rays, {int(np.sum(run[0] >= 0))} hits, {len(diff)} differ in the grazing band")
    return len(diff)


def _check_boxes(tris, lo, hi, child, order):
    """The invariants of test_tree_invariants: child boxes nest in their parent's slot, leaf boxes contain the widened
    triangles."""
    n = len(tris)
    v = tris[:, :9].reshape(-1, 3, 3)
    for node in range(max(n - 1, 1)):
        for side in range(2):
            c = child[node, side]
            if c >= 0:
                assert np.all(lo[c].min(0) >= lo[node, side]) and np.all(hi[c].max(0) <= hi[node, side])
            else:
                t = v[order[~c]]
                mn, mx = t.min(0), t.max(0)
                w = (mx - mn) * np.float32(2.0e-4)
                assert np.all(lo[node, side] <= mn - w) and np.all(hi[node, side] >= mx + w)


def _call(ctx, scene, mesh_index, ptr, n, flags):
    return ctx._lib.rtb_scene_mesh_update(ctx._h, scene._h, mesh_index, C.c_void_p(ptr), n, flags, None)


# ---- rebuild ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("model", ["ball", "torus100k", "one_triangle"])
def test_rebuild_equals_fresh_upload(ctx, model):
    tris = _model(model)
    new = twist(tris, 0.6, 1.05)
    s, fresh = ctx.upload(_flat(tris, True, lead_sphere=False)), ctx.upload(_flat(new, True, lead_sphere=False))
    try:
        s.mesh_update(new)
        assert _tree_bytes(s) == _tree_bytes(fresh)
        rays = _all_rays(new, 21)
        assert _hits(s, rays) == _hits(fresh, rays)
    finally:
        s.close()
        fresh.close()


def _preset3_pair(deformed):
    """(mesh preset 3 with the STL's records, a preset 3 whose loose records are `deformed`: the fresh-upload reference)."""
    a = _preset3(True)
    b = _preset3(True)
    f = b.flat.contents
    np.ctypeslib.as_array(f.loose_tri, shape=(f.n_loose * 12,))[:] = deformed.ravel()
    return a, b


@pytest.mark.gpu
def test_rebuild_preset3_images_equal_fresh_upload(ctx):
    ball = _ball()  # the STL records preset 3 loads
    new = twist(ball, 0.8, 1.1)
    a, b = _preset3_pair(new)
    da, db = ctx.upload(a.flat), ctx.upload(b.flat)
    try:
        da.mesh_update(new)
        for setting in (a.setting, rtb200.make_setting("simple")):
            frame = rtb200.make_frame(400, 300, samples=4, seed=7, counters=1)
            (ia, sa), (ib, sb) = da.render(a.camera, setting, frame), db.render(b.camera, setting, frame)
            assert ia.tobytes() == ib.tobytes() and sa["n_rays"] == sb["n_rays"]
    finally:
        da.close()
        db.close()
        a.close()
        b.close()


# ---- refit --------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("model", ["ball", "torus100k", "one_triangle"])
def test_refit_keeps_the_shape_and_the_contract(ctx, model):
    tris = _model(model)
    new = twist(tris, 0.6, 1.05)
    s, run = ctx.upload(_flat(tris, True, lead_sphere=False)), ctx.upload(_flat(new, False, lead_sphere=False))
    try:
        before = _tree_bytes(s)
        s.mesh_update(tris, refit=True)
        assert _tree_bytes(s) == before, "a refit with the same records changed the tree"
        s.mesh_update(new, refit=True)
        lo, hi, child, order, depth = s.mesh_download()
        assert child.tobytes() == before[2] and order.tobytes() == before[3] and depth == before[4]
        _check_boxes(new, lo, hi, child, order)
        rays = _all_rays(new, 22)
        _band_only(new, rays, run.intersect_rays(rays), s.intersect_rays(rays), f"refit {model}")
    finally:
        s.close()
        run.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["mc", "simple_tree", "chain"])
def test_refit_preset3_images_equal_run(ctx, kind):
    setting = None if kind == "mc" else rtb200.make_setting("simple")
    run = _preset3(False)
    ball = _loose(run.flat).reshape(-1, 12)
    new = twist(ball, 0.8, 1.1)
    f = run.flat.contents
    np.ctypeslib.as_array(f.loose_tri, shape=(f.n_loose * 12,))[:] = new.ravel()
    mesh = _preset3(True)
    if kind == "chain":
        _material_non_refractive(run)
        _material_non_refractive(mesh)
    dr, dm = ctx.upload(run.flat), ctx.upload(mesh.flat)
    try:
        dm.mesh_update(new, refit=True)
        frame = rtb200.make_frame(400, 300, samples=4, seed=7, counters=1)
        (ir, sr), (im, sm) = dr.render(run.camera, setting or run.setting, frame), dm.render(mesh.camera, setting or mesh.setting, frame)
        assert ir.tobytes() == im.tobytes(), f"{kind}: refitted mesh image differs from the run's"
        assert sr["n_rays"] == sm["n_rays"]
    finally:
        dr.close()
        dm.close()
        run.close()
        mesh.close()


# ---- device source and ordering -----------------------------------------------------------------
def _twist_torch(t, amount, scale):
    """twist() in torch ops on the device (float32 throughout: the records differ from twist()'s, which is fine -- the
    host comparison copies these very records back)."""
    import torch
    v = t[:, :9].reshape(-1, 3)
    lo, hi = v.min(0).values, v.max(0).values
    c = (lo + hi) / 2
    p = (v - c) * scale
    a = amount * (v[:, 1] - lo[1]) / (hi[1] - lo[1])
    x = p[:, 0] * torch.cos(a) - p[:, 2] * torch.sin(a)
    z = p[:, 0] * torch.sin(a) + p[:, 2] * torch.cos(a)
    w = (torch.stack([x, p[:, 1], z], 1) + c).reshape(-1, 3, 3)
    n = torch.linalg.cross(w[:, 1] - w[:, 0], w[:, 2] - w[:, 0])
    n = n / n.norm(dim=1, keepdim=True).clamp_min(1e-30)
    return torch.cat([w.reshape(-1, 9), n], 1).contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("refit", [False, True])
def test_device_source_equals_host_source(ctx, refit):
    import torch
    tris = _tris_from_facets(rtb200.torus_triangles(1_000_000, seed=6))
    f = _flat(tris, True, lead_sphere=False)
    sd, sh = ctx.upload(f), ctx.upload(f)
    try:
        side = torch.cuda.Stream(device=0)
        with torch.cuda.stream(side):
            t = torch.from_numpy(tris).to("cuda:0", non_blocking=False)
            for _ in range(8):  # enough work on the side stream that a missing wait would read unfinished records
                t = _twist_torch(t, 0.05, 1.0)
            sd.mesh_update(t, refit=refit)  # no synchronise: ordered behind the side stream
        side.synchronize()
        host = t.cpu().numpy()
        sh.mesh_update(host, refit=refit)
        assert _tree_bytes(sd) == _tree_bytes(sh)
        rays = _all_rays(host, 23, 512)
        assert _hits(sd, rays) == _hits(sh, rays)
    finally:
        sd.close()
        sh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("refit", [False, True])
def test_device_source_on_torchs_default_stream(ctx, refit):
    """Records produced by torch ops on torch's default stream, no synchronise before the call, and overwritten in place on
    that stream right after it: the update reads them after the ops that produce them and before the overwrite."""
    import torch
    tris = _tris_from_facets(rtb200.torus_triangles(1_000_000, seed=6))
    f = _flat(tris, True, lead_sphere=False)
    sd, sh = ctx.upload(f), ctx.upload(f)
    try:
        torch.cuda.synchronize()
        with torch.cuda.stream(torch.cuda.default_stream(0)):
            t = torch.from_numpy(tris).to("cuda:0")
            for _ in range(8):
                t = _twist_torch(t, 0.05, 1.0)
            expected = t.clone()
            sd.mesh_update(t, refit=refit)
            t.mul_(3.0)  # the next "simulation step" writes the records in place
        torch.cuda.synchronize()
        host = expected.cpu().numpy()
        sh.mesh_update(host, refit=refit)
        assert _tree_bytes(sd) == _tree_bytes(sh)
        rays = _all_rays(host, 28, 512)
        assert _hits(sd, rays) == _hits(sh, rays)
    finally:
        sd.close()
        sh.close()


@pytest.mark.gpu
def test_misaligned_device_records_are_rejected(ctx):
    import torch
    tris = _ball()
    s = ctx.upload(_flat(tris, True, lead_sphere=False))
    try:
        rays = _all_rays(tris, 24, 256)
        before, tree = _hits(s, rays), _tree_bytes(s)
        buf = torch.zeros(tris.size + 1, dtype=torch.float32, device="cuda:0")
        buf[1:] = torch.from_numpy(twist(tris, 0.5).ravel()).cuda()
        sl = buf[1:].view(-1, 12)
        torch.cuda.synchronize()
        assert _call(ctx, s, 0, sl.data_ptr(), len(tris), rtb200.MESH_REBUILD) == ERR_INVALID
        with pytest.raises(rtb200.RtbError):
            s.mesh_update(sl)
        assert _hits(s, rays) == before and _tree_bytes(s) == tree
    finally:
        s.close()


@pytest.mark.gpu
def test_update_is_ordered_between_renders_on_other_streams(ctx):
    import torch
    ball = _ball()  # the STL records preset 3 loads
    new = twist(ball, 0.8, 1.1)
    a, b = _preset3_pair(new)
    frame = rtb200.make_frame(400, 300, samples=4, seed=7)
    refs = []
    for p in (a, b):  # fresh uploads: before and after the change
        d = ctx.upload(p.flat)
        out = torch.zeros((300, 400, 3), dtype=torch.float32, device="cuda:0")
        d.render_device(p.camera, p.setting, frame, out.data_ptr())
        torch.cuda.synchronize()
        refs.append(out.cpu().numpy().tobytes())
        d.close()
    d = ctx.upload(a.flat)
    try:
        sa, sb = torch.cuda.Stream(device=0), torch.cuda.Stream(device=0)
        out1 = torch.zeros((300, 400, 3), dtype=torch.float32, device="cuda:0")
        out2 = torch.zeros((300, 400, 3), dtype=torch.float32, device="cuda:0")
        torch.cuda.synchronize()
        d.render_device(a.camera, a.setting, frame, out1.data_ptr(), stream=sa.cuda_stream)
        with torch.cuda.stream(sb):
            rec = torch.from_numpy(new).to("cuda:0")
            d.mesh_update(rec)
        d.render_device(a.camera, a.setting, frame, out2.data_ptr(), stream=sa.cuda_stream)
        torch.cuda.synchronize()
        assert out1.cpu().numpy().tobytes() == refs[0], "the frame before the update saw the new triangles"
        assert out2.cpu().numpy().tobytes() == refs[1], "the frame after the update did not see the new triangles"
    finally:
        d.close()
        a.close()
        b.close()


# ---- overlapping records, errors ------------------------------------------------------------------
def _overlap_layout(n):
    return [(0, 300), (200, n - 200), (100, 150), (0, n)]  # a run, then mesh records 0, 1, 2


@pytest.mark.gpu
@pytest.mark.parametrize("refit", [False, True])
def test_update_of_an_enclosing_record_updates_the_records_inside(ctx, refit):
    tris = _ball()
    n = len(tris)
    new = twist(tris, 0.7, 1.05)
    layout = _overlap_layout(n)
    mesh_rec = lambda t: _flat_records(t, [(rtb200.PRIM_TRIANGLES, 0, 300)] + [(rtb200.PRIM_MESH, a, c) for a, c in layout[1:]])
    s = ctx.upload(mesh_rec(tris))
    ref = ctx.upload(mesh_rec(new) if not refit else _flat_records(new, [(rtb200.PRIM_TRIANGLES, a, c) for a, c in layout]))
    try:
        s.mesh_update(new, mesh_index=2, refit=refit)
        rays = _all_rays(new, 25)
        if refit:
            _band_only(new, rays, ref.intersect_rays(rays), s.intersect_rays(rays), "refit of overlapping records")
        else:
            assert _hits(s, rays) == _hits(ref, rays)
            for j in range(3):
                assert _tree_bytes(s, j) == _tree_bytes(ref, j)
    finally:
        s.close()
        ref.close()


@pytest.mark.gpu
def test_update_of_a_partly_overlapped_record_is_refused(ctx):
    tris = _ball()
    n = len(tris)
    layout = _overlap_layout(n)
    s = ctx.upload(_flat_records(tris, [(rtb200.PRIM_TRIANGLES, 0, 300)] + [(rtb200.PRIM_MESH, a, c) for a, c in layout[1:]]))
    try:
        rays = _all_rays(tris, 26, 512)
        before, trees = _hits(s, rays), [_tree_bytes(s, j) for j in range(3)]
        new = twist(tris, 0.7)[200:]
        for flags in (rtb200.MESH_REBUILD, rtb200.MESH_REFIT):
            assert _call(ctx, s, 0, new.ctypes.data, len(new), flags) == ERR_UNSUPPORTED
        assert _hits(s, rays) == before and [_tree_bytes(s, j) for j in range(3)] == trees
    finally:
        s.close()


@pytest.mark.gpu
def test_rejected_updates_leave_the_scene_unchanged(ctx):
    import torch
    tris = _ball()
    new = twist(tris, 0.7)
    s = ctx.upload(_flat(tris, True))
    plain = ctx.upload(_flat_records(tris, [(rtb200.PRIM_TRIANGLES, 0, len(tris))]))
    try:
        rays = _all_rays(tris, 27, 512)
        before, tree, plain_before = _hits(s, rays), _tree_bytes(s), _hits(plain, rays)
        assert _call(ctx, s, 0, new.ctypes.data, len(new) - 1, rtb200.MESH_REBUILD) == ERR_INVALID  # wrong n
        assert _call(ctx, s, 1, new.ctypes.data, len(new), rtb200.MESH_REBUILD) == ERR_UNSUPPORTED  # no such mesh
        assert _call(ctx, s, -1, new.ctypes.data, len(new), rtb200.MESH_REFIT) == ERR_UNSUPPORTED
        assert _call(ctx, s, 0, new.ctypes.data, len(new), 7) == ERR_INVALID  # unknown flags
        assert _call(ctx, plain, 0, new.ctypes.data, len(new), rtb200.MESH_REBUILD) == ERR_UNSUPPORTED  # a scene without a mesh
        if torch.cuda.device_count() >= 2:
            other = torch.from_numpy(new).to("cuda:1")
            torch.cuda.synchronize(1)
            assert _call(ctx, s, 0, other.data_ptr(), len(new), rtb200.MESH_REBUILD) == ERR_INVALID  # another device's memory
        assert _hits(s, rays) == before and _tree_bytes(s) == tree and _hits(plain, rays) == plain_before
    finally:
        s.close()
        plain.close()


# ---- several devices ----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("refit", [False, True])
def test_multi_scene_update_equals_single_device(ctx, refit):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two or more GPUs")
    p = _preset3(True)
    new = twist(_loose(p.flat).reshape(-1, 12), 0.8, 1.1)
    frame = rtb200.make_frame(400, 300, samples=4, seed=7)
    m = rtb200.MultiContext(2)
    try:
        ms, d = m.upload(p.flat), ctx.upload(p.flat)
        try:
            ms.mesh_update(new, refit=refit)
            d.mesh_update(new, refit=refit)
            img_m, st_m = ms.render(p.camera, p.setting, frame)
            img_s, st_s = d.render(p.camera, p.setting, frame)
        finally:
            ms.close()
            d.close()
        assert img_m.tobytes() == img_s.tobytes() and st_m["n_rays"] == st_s["n_rays"]
    finally:
        m.close()
        p.close()


def test_header_flags_match_the_bindings():
    import os
    import re
    text = open(os.path.join(rtb200.ROOT, "include", "rtb.h")).read()
    assert re.search(r"enum \{ RTB_MESH_REBUILD = 0, RTB_MESH_REFIT = 1 \};", text)
    assert (rtb200.MESH_REBUILD, rtb200.MESH_REFIT) == (0, 1)
    assert {"rtb_scene_mesh_update", "rtb_multi_scene_mesh_update"} <= set(rtb200.ABI_SYMBOLS)
