"""Closest-point queries on device buffers (rtb_query_points), on the GPU.

Scenes: seeded tori (rtb200.torus_triangles, tube radius 6) of 10 k, 100 k and 1 M triangles as a MESH record, preset 3's
ball (528 triangles) as a mesh, and -- the in-library brute force the hierarchy is measured against -- the 10 k and 100 k tori
as a TRIANGLES run.  Point sets, made by torch ops on the device:

  near:          on uniformly drawn triangles (barycentric), moved along the normal by up to +-1 % of the tube radius
                 (the ball: of its half extent), in triangle order -- the tori's triangles are laid out ring by ring, so
                 neighbouring points are neighbours in space;
  near_shuffled: the same points in random order (what spatial coherence is worth);
  uniform:       uniform in the model's bounding box.

Modes: closest unbounded, closest bounded (radius 5 % of the tube radius), any with the same radius.  CUDA-event ms of one
call on a side stream with preallocated outputs, the median of --reps after a warm-up; the inputs of the 16 Mi sets (256 MB of
points and outputs) do not fit the 126 MB L2.  The brute-force runs are measured only up to 1e10 point-triangle pairs.

The twist sequence: tools/mesh_update_probe.py's 30-step large twist of the 1 M-triangle torus, each step a refit from device
records followed by 64 Ki closest queries and 64 Ki any queries on the same stream, one synchronise per step; host clock per
step, summed.

The GPU name, power limit and max SM clock are read in the same call.

    python tools/point_query_probe.py --out profiles/r06_point_query_probe.json
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np
import torch

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rtb200  # noqa: E402
from mesh_probe import gpu_info  # noqa: E402
from mesh_update_probe import twist_device  # noqa: E402
from ray_query_probe import event_ms  # noqa: E402


def flat_scene(tris, prim_type):
    """one record of `tris` ([n][12] a, b, c, normal) as a MESH or TRIANGLES record"""
    tris = np.ascontiguousarray(tris, np.float32)
    mats = (rtb200.Material * 1)()
    mats[0].diffusiveness = 1.0
    prims = (rtb200.Prim * 1)()
    prims[0].type, prims[0].count = prim_type, len(tris)
    f = rtb200.FlatScene()
    f.n_prims, f.prims, f.n_materials, f.materials = 1, prims, 1, mats
    f.n_top, f.n_loose = len(tris), len(tris)
    f.loose_tri = tris.ctypes.data_as(C.POINTER(C.c_float))
    f._keep = (tris, mats, prims)
    return f


def torus(n):
    f = rtb200.torus_triangles(n, seed=n)
    return np.concatenate([f[:, 3:12], f[:, :3]], 1).astype(np.float32)


def ball():
    s = rtb200.PresetScene(3)
    try:
        f = s.flat.contents
        return np.ctypeslib.as_array(f.loose_tri, shape=(f.n_loose, 12)).copy()
    finally:
        s.close()


def point_sets(tris, n, scale, seed):
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    t = torch.from_numpy(tris).cuda()
    k = torch.randint(0, len(tris), (n,), device="cuda:0", generator=g).sort().values
    w = torch.rand(n, 3, device="cuda:0", generator=g)
    w = w / w.sum(1, keepdim=True)
    v = t[k, :9].reshape(n, 3, 3)
    near = (w[:, :, None] * v).sum(1) + t[k, 9:12] * ((torch.rand(n, 1, device="cuda:0", generator=g) * 2 - 1) * 0.01 * scale)
    lo, hi = t[:, :9].reshape(-1, 3).min(0).values, t[:, :9].reshape(-1, 3).max(0).values
    uniform = lo + torch.rand(n, 3, device="cuda:0", generator=g) * (hi - lo)
    perm = torch.randperm(n, device="cuda:0", generator=g)
    return {"near": near.contiguous(), "near_shuffled": near[perm].contiguous(), "uniform": uniform.contiguous()}


def measure(d, tris, n, scale, stream, reps):
    sets = point_sets(tris, n, scale, n)
    out_c = (torch.empty(n, dtype=torch.int32, device="cuda:0"), torch.empty(n, device="cuda:0"),
             torch.empty(n, 3, device="cuda:0"), torch.empty(n, 3, device="cuda:0"))
    out_a = torch.empty(n, dtype=torch.bool, device="cuda:0")
    r = 0.05 * scale
    res = dict(points=n, radius=r)
    torch.cuda.synchronize()
    for kind, pts in sets.items():
        e = dict()
        e["closest_unbounded_ms"] = event_ms(lambda: d.closest_points(pts, out=out_c, stream=stream.cuda_stream), stream, reps)
        e["median_distance"] = float(out_c[1].median())
        e["closest_bounded_ms"] = event_ms(lambda: d.closest_points(pts, max_dist=r, out=out_c, stream=stream.cuda_stream), stream, reps)
        e["hit_fraction_bounded"] = float((out_c[0] >= 0).float().mean())
        e["any_ms"] = event_ms(lambda: d.closest_points(pts, max_dist=r, any_hit=True, out=out_a, stream=stream.cuda_stream), stream, reps)
        res[kind] = e
    return res


def twist_sequence(ctx, tris, steps, twist, npts, scale, stream):
    d = ctx.upload(flat_scene(tris, rtb200.PRIM_MESH))
    base = torch.from_numpy(tris).cuda()
    pts = point_sets(tris, npts, scale, 1)["near"]  # near the untwisted surface: the twist moves the surface away from some
    step_ms = []
    try:
        for k in range(steps + 1):  # step 0: warm-up
            rec = twist_device(base, twist * max(k, 1) / steps)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with torch.cuda.stream(stream):
                d.mesh_update(rec, refit=True)
                d.closest_points(pts)
                d.closest_points(pts, max_dist=0.05 * scale, any_hit=True)
            stream.synchronize()
            if k:
                step_ms.append((time.perf_counter() - t0) * 1e3)
    finally:
        d.close()
    return dict(step_ms_sum=sum(step_ms), step_ms_median=float(np.median(step_ms)), step_ms=[round(x, 4) for x in step_ms])


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--sizes", default="4096,262144,16777216")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--twist", type=float, default=1.5)
    ap.add_argument("--step-points", type=int, default=65536)
    a = ap.parse_args()
    ctx = rtb200.Context(0)
    stream = torch.cuda.Stream(device=0)
    res = dict(gpu=gpu_info(), workloads=[])
    b = ball()
    bv = b[:, :9].reshape(-1, 3)
    jobs = [("torus_10k_mesh", torus(10_000), rtb200.PRIM_MESH, 6.0), ("torus_100k_mesh", torus(100_000), rtb200.PRIM_MESH, 6.0),
            ("torus_1m_mesh", torus(1_000_000), rtb200.PRIM_MESH, 6.0),
            ("ball_mesh", b, rtb200.PRIM_MESH, float((bv.max(0) - bv.min(0)).max() / 2)),
            ("torus_10k_run", torus(10_000), rtb200.PRIM_TRIANGLES, 6.0), ("torus_100k_run", torus(100_000), rtb200.PRIM_TRIANGLES, 6.0)]
    for name, tris, typ, scale in jobs:
        d = ctx.upload(flat_scene(tris, typ))
        for n in [int(x) for x in a.sizes.split(",") if x]:
            if typ == rtb200.PRIM_TRIANGLES and n * len(tris) > 1e10:
                continue
            entry = dict(workload=name, triangles=len(tris), **measure(d, tris, n, scale, stream, a.reps if n < (1 << 24) else 3))
            print(json.dumps(entry), flush=True)
            res["workloads"].append(entry)
        d.close()
    r = twist_sequence(ctx, torus(1_000_000), a.steps, a.twist, a.step_points, 6.0, stream)
    res["twist_sequence"] = dict(steps=a.steps, twist=a.twist, points_per_step=a.step_points, mode="refit", **r)
    print(json.dumps({k: v for k, v in res["twist_sequence"].items() if k != "step_ms"}), flush=True)
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
