"""rtb_query_triangles: which of the scene's TRIANGLES and MESH triangles a batch of query triangles shares a point with,
decided exactly, on device buffers and ordered on the caller's stream (include/rtb.h, DESIGN 3g).  Oracles: an independent
exact separating-axis test in Python integers (from fractions.Fraction), the overlap test csrc/rtb_tritri.h compiled for the
host (its CPU check, and a brute-force loop over it), and for mesh records the run of the same triangles.  GPU results are
compared as exact sets (multisets where overlapping records report a triangle twice); there are no tolerances."""
import ctypes as C
import os
import re
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import rtb200
from rtb200 import PresetScene
from test_mesh import _ball, _flat, _flat_records, _preset3, _tris_from_facets
from test_mesh_update import _overlap_layout, twist
from test_point_query import _packed

ERR_INVALID = -1
CSRC = os.path.join(rtb200.PKG, "csrc")


# ---- host side (no device) --------------------------------------------------------------------
def _check_exe(tmp_path):
    exe = str(tmp_path / "tritri_check")
    src = os.path.join(rtb200.ROOT, "tests", "tritri_check.cpp")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-o", exe, src])
    return exe


def _counts(stdout):
    return {k: int(v) for k, v in re.findall(r"(\w+) (\d+)", stdout.splitlines()[-1])}


def test_tritri_check_on_the_cpu(tmp_path):
    """csrc/rtb_tritri.h for the host over random and adversarial pairs: degenerate triangles intersect nothing, box-separated
    pairs do not intersect (the pruning lemma), the answer is invariant under swapping and reordering, constructed contacts
    are found, and the adversarial sets run the exact fallback heavily."""
    exe = _check_exe(tmp_path)
    for seed in (1, 2):
        out = subprocess.run([exe, str(seed), "200000"], capture_output=True, text=True)
        print(out.stdout)
        assert out.returncode == 0, out.stdout
        c = _counts(out.stdout)
        assert c["violations"] == 0 and c["checked"] == 200000
        assert c["fallback_pairs"] > 50000 and c["exact3"] > 100000 and c["exact2"] > 10000
        assert 20000 < c["intersecting"] < 180000 and c["degenerate"] > 20000


def _oracle_ints(p, q):
    """the 18 coordinates as integers on one dyadic scale (exact: every float is an integer times a power of two)"""
    fr = [Fraction(float(x)) for x in list(p) + list(q)]
    den = max(f.denominator for f in fr)
    return [int(f * den) for f in fr]


def _oracle_degenerate(v):
    if not all(np.isfinite(v)):
        return True
    x = [Fraction(float(c)) for c in v]
    u = [x[3 + i] - x[i] for i in range(3)]
    w = [x[6 + i] - x[i] for i in range(3)]
    return u[1] * w[2] - u[2] * w[1] == 0 and u[2] * w[0] - u[0] * w[2] == 0 and u[0] * w[1] - u[1] * w[0] == 0


def _oracle(p, q):
    """exact: two non-degenerate closed triangles are disjoint exactly when one of these axes strictly separates them: the two
    normals, the nine edge-edge cross products and the six in-plane edge normals n x e (zero axes skipped)"""
    if _oracle_degenerate(p) or _oracle_degenerate(q):
        return False
    v = _oracle_ints(p, q)
    P, Q = [v[0:3], v[3:6], v[6:9]], [v[9:12], v[12:15], v[15:18]]
    sub = lambda a, b: [a[0] - b[0], a[1] - b[1], a[2] - b[2]]
    cross = lambda a, b: [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]
    dot = lambda a, b: a[0] * b[0] + a[1] * b[1] + a[2] * b[2]
    ep = [sub(P[1], P[0]), sub(P[2], P[1]), sub(P[0], P[2])]
    eq = [sub(Q[1], Q[0]), sub(Q[2], Q[1]), sub(Q[0], Q[2])]
    n1, n2 = cross(ep[0], ep[1]), cross(eq[0], eq[1])
    for ax in [n1, n2] + [cross(a, b) for a in ep for b in eq] + [cross(n1, e) for e in ep] + [cross(n2, e) for e in eq]:
        if ax == [0, 0, 0]:
            continue
        a, b = [dot(ax, x) for x in P], [dot(ax, x) for x in Q]
        if max(a) < min(b) or max(b) < min(a):
            return False
    return True


def test_fraction_oracle_basics():
    t = [0, 0, 0, 1, 0, 0, 0, 1, 0]
    assert _oracle(t, [1, 0, 0, 2, 0, 0, 1, 1, 0])  # a shared vertex
    assert not _oracle(t, [0, 0, 1, 1, 0, 1, 0, 1, 1])  # parallel planes
    assert _oracle(t, [0.25, 0.25, -1, 0.25, 0.25, 1, 3, 3, 0])  # an edge through the face
    assert not _oracle(t, [0.5, 0.5 + 2 ** -24, 0, 2, 2, 0, 0.5 + 2 ** -23, 2, 0])  # coplanar, one ulp beyond the hypotenuse
    assert _oracle(t, [0.5, 0.5, 0, 2, 2, 0, 0.5, 2, 0])  # coplanar, touching the hypotenuse
    assert not _oracle(t, [0, 0, 0, 2, 0, 0, 4, 0, 0])  # collinear: degenerate


_HOST_SRC = r"""
#include "rtb_tritri.h"
// the header on raw pairs p[n][9], q[n][9]
extern "C" void tri_batch(const float *p, const float *q, long n, unsigned char *out)
{
    for (long i = 0; i < n; i++) out[i] = rtb_tritri::intersect(p + 9 * i, q + 9 * i);
}
// brute force: query triangles qt[n][12] (a, b, c, n) against packed records t[m][12] (a, a - b, a - c, n) as one TRIANGLES run
// with ids base + k; every pair (i, base + k) is written while fewer than cap, the total returned
extern "C" long tri_pairs(const float *qt, long n, const float *t, long m, int base, int *out, long cap)
{
    long cnt = 0;
    for (long i = 0; i < n; i++)
    {
        const float *p = qt + 12 * i;
        if (rtb_tritri::degenerate(p)) continue;
        float lo[3], hi[3], tlo[3], thi[3];
        rtb_tritri::box(p, lo, hi);
        for (long k = 0; k < m; k++)
        {
            const float *r = t + 12 * k;
            const float v[9] = {r[0], r[1], r[2], r[0] - r[3], r[1] - r[4], r[2] - r[5], r[0] - r[6], r[1] - r[7], r[2] - r[8]};
            rtb_tritri::box(v, tlo, thi);
            if (!rtb_tritri::boxesOverlap(lo, hi, tlo, thi) || !rtb_tritri::meets(p, v)) continue;
            if (cnt < cap) { out[2 * cnt] = (int)i; out[2 * cnt + 1] = base + (int)k; }
            cnt++;
        }
    }
    return cnt;
}
"""


@pytest.fixture(scope="module")
def host_model(tmp_path_factory):
    d = tmp_path_factory.mktemp("tritri_host")
    src, so = d / "tritri_host.cpp", d / "tritri_host.so"
    src.write_text(_HOST_SRC)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-I", CSRC, "-o", str(so), str(src)])
    lib = C.CDLL(str(so))
    vp = C.c_void_p
    lib.tri_batch.argtypes = [vp, vp, C.c_long, vp]
    lib.tri_pairs.argtypes = [vp, C.c_long, vp, C.c_long, C.c_int, vp, C.c_long]
    lib.tri_pairs.restype = C.c_long
    return lib


def test_header_agrees_with_the_fraction_oracle(tmp_path, host_model):
    """Every pair of a dump of the check's generators -- random, contacts, coplanar, one ulp off, offsets, denormals,
    degenerate; every pair that took the exact fallback included -- is decided alike by the host-compiled header and the
    exact oracle."""
    exe, dump = _check_exe(tmp_path), str(tmp_path / "pairs.bin")
    out = subprocess.run([exe, "3", "30000", dump], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    rec = np.fromfile(dump, np.dtype([("p", "<f4", 9), ("q", "<f4", 9), ("hit", "u1"), ("fell", "u1"), ("kind", "u1")]))
    assert len(rec) == 30000
    p, q = np.ascontiguousarray(rec["p"]), np.ascontiguousarray(rec["q"])
    got = np.zeros(len(rec), np.uint8)
    host_model.tri_batch(p.ctypes.data, q.ctypes.data, len(rec), got.ctypes.data)
    assert np.array_equal(got, rec["hit"]), "the host library and the check disagree"
    exp = np.array([_oracle(a, b) for a, b in zip(p, q)])
    bad = np.nonzero(exp != got.astype(bool))[0]
    print(f"{len(rec)} pairs, {int(rec['fell'].sum())} through the exact fallback, {int(exp.sum())} intersecting")
    assert len(bad) == 0, f"{len(bad)} pairs differ from the oracle, e.g. {p[bad[0]].tolist()} {q[bad[0]].tolist()} header {got[bad[0]]}"
    assert rec["fell"].sum() > 10000
    for k in range(10):
        assert (rec["kind"] == k).sum() == 3000


def test_header_triangle_query_matches_the_bindings():
    text = open(os.path.join(rtb200.ROOT, "include", "rtb.h")).read()
    assert re.search(r"enum \{ RTB_QUERY_CLOSEST = 0, RTB_QUERY_ANY = 1 \};", text)
    assert re.search(r"\nenum \{ RTB_QUERY_PAIRS = 2 \};\n", text)
    assert re.search(r"int rtb_query_triangles\(rtb_ctx \*ctx, const rtb_scene \*scene, int64_t n, const float \*tris, int32_t flags, "
                     r"uint8_t \*hit,\s+int32_t \*pairs, int64_t capacity, int64_t \*count, void \*stream\);", text)
    assert (rtb200.QUERY_ANY, rtb200.QUERY_PAIRS) == (1, 2)
    assert "rtb_query_triangles" in rtb200.ABI_SYMBOLS
    assert "#define RTB_ABI_VERSION 5" in text


# ---- scenes and queries ------------------------------------------------------------------------
def _torus(n, seed):
    return _tris_from_facets(rtb200.torus_triangles(n, seed=seed))


def _moved(tris, angle, shift):
    """tris rotated about the x axis through the torus centre (0, 16, 0) and shifted: a second, interpenetrating torus"""
    v = tris[:, :9].reshape(-1, 3).astype(np.float64) - (0.0, 16.0, 0.0)
    c, s = np.cos(angle), np.sin(angle)
    v = np.stack([v[:, 0], c * v[:, 1] - s * v[:, 2], s * v[:, 1] + c * v[:, 2]], 1) + (0.0, 16.0, 0.0) + np.asarray(shift)
    out = tris.copy()
    out[:, :9] = v.reshape(-1, 9).astype(np.float32)
    return out


def _host_pairs(host_model, queries, tris, base=0):
    q, t = np.ascontiguousarray(queries, np.float32), _packed(tris)
    n = host_model.tri_pairs(q.ctypes.data, len(q), t.ctypes.data, len(t), base, None, 0)
    out = np.zeros((max(n, 1), 2), np.int32)
    assert host_model.tri_pairs(q.ctypes.data, len(q), t.ctypes.data, len(t), base, out.ctypes.data, n) == n
    return out[:n]


def _sorted(pairs):
    p = np.asarray(pairs, np.int64).reshape(-1, 2)
    return p[np.lexsort((p[:, 1], p[:, 0]))]


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


@pytest.fixture(scope="module")
def ctx():
    c = rtb200.Context(0)
    yield c
    c.close()


def _case(name):
    """(flat scene, [(first, count, base_id)] of its triangle records, the triangles, query triangles)"""
    if name.startswith("torus"):
        tris = _torus(10_000, 11)
        return _flat(tris, name == "torus_mesh", lead_sphere=False), [(0, len(tris), 0)], tris, _moved(_torus(4_000, 12), 0.7, (3.0, 1.0, 2.0))
    if name == "ball":
        s = _preset3(True)
        f = s.flat.contents
        recs = [(int(p.first), int(p.count), int(p.base_id)) for p in f.prims[:f.n_prims] if p.type == rtb200.PRIM_MESH]
        return s, recs, _ball(), _shifted(_ball())
    tris = _ball()
    layout = [(0, 300)] + _overlap_layout(len(tris))[1:]
    flat = _flat_records(tris, [(rtb200.PRIM_TRIANGLES, 0, 300)] + [(rtb200.PRIM_MESH, a, c) for a, c in layout[1:]])
    return flat, [(a, c, a) for a, c in layout], tris, _shifted(tris)


def _shifted(tris):
    """a twisted copy of the model moved by 30 % of its extent along x: the two surfaces cross along a closed curve"""
    out = twist(tris, 0.4)
    v = tris[:, :9].reshape(-1, 3)
    out[:, 0:9:3] += np.float32(0.3 * float(v[:, 0].max() - v[:, 0].min()))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["torus_mesh", "torus_run", "ball", "overlap"])
def test_gpu_equals_host_brute_force(ctx, host_model, name):
    """PAIRS equals a brute-force loop over the host-compiled header as a multiset (overlapping records report a triangle once
    per record); ANY is 1 exactly for the query triangles that appear in PAIRS."""
    scene, recs, tris, queries = _case(name)
    flat = scene.flat if hasattr(scene, "flat") else scene
    s = ctx.upload(flat)
    try:
        exp = _sorted(np.concatenate([_host_pairs(host_model, queries, tris[a:a + c], b) for a, c, b in recs]))
        q = _t(queries)
        got = s.intersecting_pairs(q).cpu().numpy()
        assert got.dtype == np.int64 and np.array_equal(got, _sorted(got)), "pairs are not sorted"
        assert np.array_equal(got, exp), f"{name}: {len(got)} pairs on the GPU, {len(exp)} on the host"
        hit = s.intersects(q).cpu().numpy()
        want = np.zeros(len(queries), bool)
        want[exp[:, 0]] = True
        assert np.array_equal(hit, want)
        print(f"{name}: {len(queries)} query triangles, {len(exp)} pairs, {int(want.sum())} intersecting")
        assert len(exp) > 100 and 0 < want.sum() < len(queries)
    finally:
        s.close()
        if hasattr(scene, "close"):
            scene.close()


@pytest.mark.gpu
def test_mesh_equals_run_on_a_100k_torus(ctx):
    tris = _torus(100_000, 13)
    queries = _t(_moved(_torus(20_000, 14), 0.5, (2.0, 0.5, 1.0)))
    sm, sr = ctx.upload(_flat(tris, True)), ctx.upload(_flat(tris, False))
    try:
        pm, pr = sm.intersecting_pairs(queries), sr.intersecting_pairs(queries)
        assert pm.shape[0] > 1000 and np.array_equal(pm.cpu().numpy(), pr.cpu().numpy())
        assert np.array_equal(sm.intersects(queries).cpu().numpy(), sr.intersects(queries).cpu().numpy())
    finally:
        sm.close()
        sr.close()


@pytest.mark.gpu
def test_refit_rebuild_and_fresh_upload_answer_alike(ctx):
    """After mesh_update on a side stream, with the queries enqueued right behind it, a refitted tree, a rebuilt tree and a
    fresh upload of the new triangles give the same pairs; the twist moves enough that the answer changes."""
    import torch
    tris = _torus(100_000, 15)
    new = twist(tris, 0.9, 1.05)
    queries = _t(_moved(_torus(20_000, 16), 0.5, (2.0, 0.5, 1.0)))
    refit, rebuild, fresh = ctx.upload(_flat(tris, True)), ctx.upload(_flat(tris, True)), ctx.upload(_flat(new, True))
    try:
        before = refit.intersecting_pairs(queries).cpu().numpy()
        torch.cuda.synchronize()
        st = torch.cuda.Stream(device=0)
        res = {}
        with torch.cuda.stream(st):
            rec = _t(new)
            for s, is_refit, key in ((refit, True, "refit"), (rebuild, False, "rebuild")):
                s.mesh_update(rec, refit=is_refit)
                res[key] = (s.intersects(queries), s.intersecting_pairs(queries))
        ref = (fresh.intersects(queries), fresh.intersecting_pairs(queries))
        torch.cuda.synchronize()
        assert not np.array_equal(before, ref[1].cpu().numpy())
        for key in ("refit", "rebuild"):
            assert torch.equal(res[key][0], ref[0]) and torch.equal(res[key][1], ref[1]), key
    finally:
        for s in (refit, rebuild, fresh):
            s.close()


# ---- counting and capacity ---------------------------------------------------------------------
def _raw(ctx, scene, n, tris, flags, hit=None, pairs=None, capacity=0, count=None, stream=None):
    p = lambda x: None if x is None else C.c_void_p(x if isinstance(x, int) else x.data_ptr())
    return ctx._lib.rtb_query_triangles(ctx._h, scene._h, n, p(tris), flags, p(hit), p(pairs), capacity, p(count), p(stream))


@pytest.mark.gpu
def test_capacity_overflow_and_counting_pass(ctx):
    import torch
    tris = _torus(10_000, 11)
    s = ctx.upload(_flat(tris, True, lead_sphere=False))
    try:
        q = _t(_moved(_torus(4_000, 12), 0.7, (3.0, 1.0, 2.0)))
        full = s.intersecting_pairs(q).cpu().numpy()
        total = len(full)
        cap, guard = total // 3, 1000
        buf = torch.full((cap + guard, 2), -7, dtype=torch.int32, device="cuda:0")
        count = torch.full((1,), -5, dtype=torch.int64, device="cuda:0")
        torch.cuda.synchronize()
        assert _raw(ctx, s, q.shape[0], q, rtb200.QUERY_PAIRS, pairs=buf, capacity=cap, count=count) == 0
        torch.cuda.synchronize()
        assert int(count.item()) == total
        written = buf[:cap].cpu().numpy()
        assert (buf[cap:] == -7).all(), "a slot beyond capacity was written"
        fs = {tuple(x) for x in full.tolist()}
        assert all(tuple(x) in fs for x in written.tolist()) and len({tuple(x) for x in written.tolist()}) == cap
        count.fill_(-5)
        assert _raw(ctx, s, q.shape[0], q, rtb200.QUERY_PAIRS, count=count) == 0  # counting pass
        torch.cuda.synchronize()
        assert int(count.item()) == total
        count.fill_(-5)
        assert _raw(ctx, s, 0, None, rtb200.QUERY_PAIRS, count=count) == 0  # n == 0 still defines the count
        torch.cuda.synchronize()
        assert int(count.item()) == 0
        again = s.intersecting_pairs(q, capacity=1).cpu().numpy()  # too small: a second call
        assert np.array_equal(again, full)
        assert np.array_equal(s.intersecting_pairs(q, capacity=0).cpu().numpy(), full)
    finally:
        s.close()


# ---- contact cases in a scene --------------------------------------------------------------------
def _cube(lo, hi):
    """12 outward triangles (a, b, c, normal) of the box [lo, hi]"""
    x0, y0, z0 = lo
    x1, y1, z1 = hi
    v = np.array([[x0, y0, z0], [x1, y0, z0], [x1, y1, z0], [x0, y1, z0], [x0, y0, z1], [x1, y0, z1], [x1, y1, z1], [x0, y1, z1]],
                 np.float32)
    f = [(0, 2, 1), (0, 3, 2), (4, 5, 6), (4, 6, 7), (0, 1, 5), (0, 5, 4), (2, 3, 7), (2, 7, 6), (0, 4, 7), (0, 7, 3), (1, 2, 6), (1, 6, 5)]
    t = v[np.array(f)]
    n = np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0])
    return np.concatenate([t.reshape(-1, 9), n], 1).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("mesh", [True, False])
def test_contact_cases(ctx, host_model, mesh):
    """Exactly stacked cubes (a shared face plane, shared vertices) touch; one ulp apart they do not; degenerate query triangles
    are never reported, not even on the cube's surface."""
    cube = _cube((0, 0, 0), (1, 1, 1))
    s = ctx.upload(_flat(cube, mesh, lead_sphere=False))
    try:
        up = np.nextafter(np.float32(1), np.float32(2))
        stacked, apart = _cube((0, 0, 1), (1, 1, 2)), _cube((0, 0, up), (1, 1, 2))
        side = _cube((1, 0, 0), (2, 1, 1))  # sharing the face x = 1
        corner = _cube((1, 1, 1), (2, 2, 2))  # sharing one vertex
        got = s.intersecting_pairs(_t(np.concatenate([stacked, apart, side, corner]))).cpu().numpy()
        exp = _sorted(_host_pairs(host_model, np.concatenate([stacked, apart, side, corner]), cube))
        assert np.array_equal(got, exp)
        rows = set(got[:, 0].tolist())
        assert rows & set(range(0, 12)) and rows & set(range(24, 36)) and rows & set(range(36, 48))
        assert not rows & set(range(12, 24)), "cubes one ulp apart were reported"
        deg = cube.copy()
        deg[0::4, 3:6] = deg[0::4, 0:3]  # repeated vertex
        deg[1::4, 6:9] = deg[1::4, 0:3] + 2 * (deg[1::4, 3:6] - deg[1::4, 0:3])  # collinear
        deg[2::4, 6:9] = deg[2::4, 3:6]
        deg[3::4, 4] = np.nan
        dq = _t(deg)
        assert s.intersecting_pairs(dq).shape[0] == 0 and not s.intersects(dq).any()
    finally:
        s.close()


@pytest.mark.gpu
def test_the_tunnel_is_ignored(ctx):
    s = PresetScene(5, "sah", 24)
    d = ctx.upload(s.flat)
    try:
        f = s.flat.contents
        tun = np.ctypeslib.as_array(f.tri, shape=(f.n_tris, 12)).copy()  # the tunnel's own triangles as queries
        q = _t(np.ascontiguousarray(tun[:, :12]))
        assert len(tun) > 1000
        assert d.intersecting_pairs(q).shape[0] == 0 and not d.intersects(q).any()
    finally:
        d.close()
        s.close()


# ---- streams -----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("where", ["side", "default"])
def test_triangles_from_torch_on_a_stream(ctx, where):
    """Query triangles made by torch ops on a side stream or torch's default stream, overwritten right after the call."""
    import torch
    tris = _torus(200_000, 17)
    s = ctx.upload(_flat(tris, True, lead_sphere=False))
    try:
        base = _t(_moved(_torus(100_000, 18), 0.5, (2.0, 0.5, 1.0)))
        torch.cuda.synchronize()
        st = torch.cuda.Stream(device=0) if where == "side" else torch.cuda.default_stream(0)
        with torch.cuda.stream(st):
            q = base.clone()
            for _ in range(4):  # work ahead of the query: a missing wait would read unfinished triangles
                q = (q * 1.0).contiguous()
            hit = s.intersects(q)
            count = torch.empty(1, dtype=torch.int64, device="cuda:0")
            assert _raw(ctx, s, q.shape[0], q, rtb200.QUERY_PAIRS, count=count,
                        stream=st.cuda_stream or rtb200.CUDA_STREAM_LEGACY) == 0
            q.fill_(float("nan"))
        torch.cuda.synchronize()
        exp = s.intersecting_pairs(base)
        want = torch.zeros(base.shape[0], dtype=torch.bool, device="cuda:0")
        want[exp[:, 0]] = True
        assert torch.equal(hit, want) and int(count.item()) == exp.shape[0] and exp.shape[0] > 1000
    finally:
        s.close()


@pytest.mark.gpu
def test_query_does_not_synchronise(ctx):
    import torch
    tris = _torus(100_000, 13)
    s = ctx.upload(_flat(tris, True, lead_sphere=False))
    try:
        q = _t(_moved(_torus(20_000, 14), 0.5, (2.0, 0.5, 1.0)))
        ref = s.intersects(q)
        torch.cuda.synchronize()
        st = torch.cuda.Stream(device=0)
        with torch.cuda.stream(st):
            torch.cuda._sleep(1_000_000_000)  # about half a second
            got = s.intersects(q)
            count = torch.empty(1, dtype=torch.int64, device="cuda:0")
            assert _raw(ctx, s, q.shape[0], q, rtb200.QUERY_PAIRS, count=count, stream=st.cuda_stream) == 0
        busy = not st.query()
        st.synchronize()
        assert busy, "the query call waited for its stream"
        assert torch.equal(got, ref) and int(count.item()) == s.intersecting_pairs(q).shape[0]
    finally:
        s.close()


@pytest.mark.gpu
def test_a_later_update_waits_for_the_query(ctx):
    """A query on stream A, then an update on stream B: the query sees the old triangles, a later one the new."""
    import torch
    tris = _torus(200_000, 17)
    new = twist(tris, 0.6, 1.05)
    s = ctx.upload(_flat(tris, True, lead_sphere=False))
    old_ref, new_ref = ctx.upload(_flat(tris, True, lead_sphere=False)), ctx.upload(_flat(new, True, lead_sphere=False))
    try:
        q = _t(_moved(_torus(400_000, 18), 0.5, (2.0, 0.5, 1.0)))
        rec = _t(new)
        torch.cuda.synchronize()
        sa, sb = torch.cuda.Stream(device=0), torch.cuda.Stream(device=0)
        with torch.cuda.stream(sa):
            torch.cuda._sleep(200_000_000)  # the query is still queued when the update is enqueued
            before = s.intersects(q)
        with torch.cuda.stream(sb):
            s.mesh_update(rec)
        with torch.cuda.stream(sa):
            after = s.intersects(q)
        torch.cuda.synchronize()
        assert torch.equal(before, old_ref.intersects(q)), "the query before the update"
        assert torch.equal(after, new_ref.intersects(q)), "the query after the update"
        assert not torch.equal(before, after)
    finally:
        for x in (s, old_ref, new_ref):
            x.close()


# ---- refusals ----------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refused_calls_write_nothing(ctx):
    import torch
    tris = _ball()
    s = ctx.upload(_flat(tris, True))
    try:
        qn = twist(tris, 0.4, 1.02)
        n = len(qn)
        q = _t(qn)
        hit = torch.full((n,), 77, dtype=torch.uint8, device="cuda:0")
        pairs = torch.full((n, 2), -7, dtype=torch.int32, device="cuda:0")
        count = torch.full((2,), -5, dtype=torch.int64, device="cuda:0")
        torch.cuda.synchronize()
        snap = [x.clone() for x in (hit, pairs, count)]
        ANY, PAIRS = rtb200.QUERY_ANY, rtb200.QUERY_PAIRS
        host = np.ascontiguousarray(qn)
        host_count = np.zeros(1, np.int64)
        pinned = rtb200.PinnedArray((n, 12))
        pinned.array[:] = qn
        mis = torch.zeros(n * 12 + 4, device="cuda:0", dtype=torch.float32)
        c32 = count.view(torch.int32)
        torch.cuda.synchronize()
        cases = {
            "host triangles": _raw(ctx, s, n, host.ctypes.data, ANY, hit),
            "page-locked host triangles": _raw(ctx, s, n, pinned._p.value, PAIRS, pairs=pairs, capacity=n, count=count),
            "misaligned triangles": _raw(ctx, s, n, mis[1:].data_ptr(), ANY, hit),
            "no triangles": _raw(ctx, s, n, None, ANY, hit),
            "n < 0": _raw(ctx, s, -1, q, ANY, hit),
            "n > INT32_MAX": _raw(ctx, s, 2 ** 31, q, ANY, hit),
            "capacity < 0": _raw(ctx, s, n, q, PAIRS, pairs=pairs, capacity=-1, count=count),
            "capacity without pairs": _raw(ctx, s, n, q, PAIRS, capacity=n, count=count),
            "unknown flags": _raw(ctx, s, n, q, 0, hit),
            "unknown flags 3": _raw(ctx, s, n, q, 3, pairs=pairs, capacity=n, count=count),
            "ANY without hit": _raw(ctx, s, n, q, ANY),
            "ANY with pairs": _raw(ctx, s, n, q, ANY, hit, pairs=pairs, capacity=n),
            "ANY with count": _raw(ctx, s, n, q, ANY, hit, count=count),
            "ANY with capacity": _raw(ctx, s, n, q, ANY, hit, capacity=5),
            "PAIRS without count": _raw(ctx, s, n, q, PAIRS, pairs=pairs, capacity=n),
            "PAIRS with hit": _raw(ctx, s, n, q, PAIRS, hit, pairs=pairs, capacity=n, count=count),
            "host count": _raw(ctx, s, n, q, PAIRS, count=host_count.ctypes.data),
            "host count, n == 0": _raw(ctx, s, 0, None, PAIRS, count=host_count.ctypes.data),
            "misaligned count": _raw(ctx, s, n, q, PAIRS, count=c32[1:].data_ptr()),
            "misaligned pairs": _raw(ctx, s, n, q, PAIRS, pairs=pairs.view(torch.int32).reshape(-1)[1:].data_ptr(), capacity=4,
                                     count=count),
        }
        torch.cuda.synchronize()
        pinned.close()
        for what, rc in cases.items():
            assert rc == ERR_INVALID, f"{what}: rc {rc}"
        for a, b in zip((hit, pairs, count), snap):
            assert torch.equal(a, b), "a refused call wrote its outputs"
        assert host_count[0] == 0
        assert _raw(ctx, s, 0, None, ANY, hit) == 0  # n == 0: nothing to do
        with pytest.raises(rtb200.RtbError):
            s.intersects(q.cpu())
        with pytest.raises(rtb200.RtbError):
            s.intersecting_pairs(q[:, :9].contiguous())
        with pytest.raises(rtb200.RtbError):
            s.intersects(q, out=torch.zeros(n + 1, dtype=torch.bool, device="cuda:0"))
    finally:
        s.close()
