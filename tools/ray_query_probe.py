"""Ray queries on device buffers (rtb_query_rays) against the host-array path (rtb_intersect_rays), on the GPU.

Scenes: a seeded torus of about 1 M triangles and preset 3's ball, both loaded through preset 3's STL path as a mesh, and
preset 5's tunnel under the k-d SAH tree (150 segments).  Ray counts: 4 Ki, 64 Ki, 1 Mi and 16 Mi.  Ray kinds:

  primary: camera rays through uniformly drawn points of the image plane, made by torch ops on the device.  The bounded
           queries take a per-ray bound drawn uniformly in [0, 2 m), m = the median unbounded hit distance.
  shadow:  from the primary rays' hit points towards a point light (beside and above the camera, m away from the eye), with
           tmax = the distance to the light.  Rays whose primary ray missed start at the eye.

Per scene, ray count and kind: CUDA-event ms of one query call on a side stream (closest unbounded, closest bounded, any;
outputs preallocated, the median of --reps after a warm-up), and the host clock of one rtb_intersect_rays call with host
arrays (rays staged in, results copied out, synchronised).  Also the fraction of hits / occluded rays.

The twist sequence redoes tools/mesh_update_probe.py's 30-step large twist of the 1 M-triangle torus with 4096 queries per
step: each step updates the mesh from device records and then queries rays from the device on the same stream (closest,
then any with the distance to a light), synchronising once at the end of the step; against the same steps with the queries
through rtb_intersect_rays.  Host clock per step.

The GPU name, power limit and max SM clock are read in the same call.

    python tools/ray_query_probe.py --out profiles/r05_ray_query_probe.json
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rtb200  # noqa: E402
from mesh_probe import gpu_info, scene  # noqa: E402
from mesh_update_probe import twist_device  # noqa: E402


def camera_rays(cam, n, seed):
    """[n][6] rays of Camera.cpp:20-26 through uniformly drawn image-plane points (float32 torch ops on the device)"""
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    sx = torch.rand(n, 1, device="cuda:0", generator=g) * 2 * cam.xcenter
    sy = torch.rand(n, 1, device="cuda:0", generator=g)
    t = lambda v: torch.tensor(list(v), dtype=torch.float32, device="cuda:0")
    v = t(cam.front) + t(cam.right) * ((sx - cam.xcenter) * cam.fov_scale) + t(cam.up) * ((sy - 0.5) * cam.fov_scale)
    d = v / v.norm(dim=1, keepdim=True)
    return torch.cat([t(cam.eye) + d * cam.forward, d], 1).contiguous()


def shadow_rays(cam, rays, hit_t, pos, m):
    light = torch.tensor(list(cam.eye), device="cuda:0") + (torch.tensor(list(cam.right), device="cuda:0") * 0.5 +
                                                           torch.tensor(list(cam.up), device="cuda:0")) * m
    o = torch.where((hit_t > 0)[:, None], pos, rays[:, :3])
    d = light - o
    dist = d.norm(dim=1)
    return torch.cat([o, d / dist[:, None]], 1).contiguous(), dist.contiguous()


def event_ms(fn, stream, reps):
    fn()  # warm-up
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            fn()
            e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms))


def host_ms(fn, reps):
    fn()
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ms.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ms))


def measure(d, cam, n, stream, reps):
    with torch.cuda.stream(stream):
        rays = camera_rays(cam, n, n)
        closest = d.query(rays)
    stream.synchronize()
    hit_t = closest[1]
    m = float(hit_t[hit_t > 0].median()) if bool((hit_t > 0).any()) else 1.0
    g = torch.Generator(device="cuda:0").manual_seed(n + 1)
    bound = (torch.rand(n, device="cuda:0", generator=g) * 2 * m).contiguous()
    srays, sdist = shadow_rays(cam, rays, hit_t, closest[2], m)
    torch.cuda.synchronize()
    out_c = tuple(torch.empty_like(x) for x in closest)
    out_a = torch.empty(n, dtype=torch.bool, device="cuda:0")
    res = dict(rays=n, median_hit_t=m)
    for kind, r, b in (("primary", rays, bound), ("shadow", srays, sdist)):
        e = dict()
        e["closest_unbounded_ms"] = event_ms(lambda: d.query(r, out=out_c, stream=stream.cuda_stream), stream, reps)
        e["hit_fraction_unbounded"] = float((out_c[0] >= 0).float().mean())
        e["closest_bounded_ms"] = event_ms(lambda: d.query(r, tmax=b, out=out_c, stream=stream.cuda_stream), stream, reps)
        e["hit_fraction_bounded"] = float((out_c[0] >= 0).float().mean())
        e["any_ms"] = event_ms(lambda: d.query(r, tmax=b, any_hit=True, out=out_a, stream=stream.cuda_stream), stream, reps)
        e["occluded_fraction"] = float(out_a.float().mean())
        host = r.cpu().numpy()
        e["intersect_rays_host_ms"] = host_ms(lambda: d.intersect_rays(host), max(1, reps // 3))
        res[kind] = e
    return res


def twist_sequence(ctx, s, base, twist, steps, nrays, stream, refit, device_queries):
    f = s.flat.contents
    np.ctypeslib.as_array(f.loose_tri, shape=(f.n_loose * 12,))[:] = base.cpu().numpy().ravel()
    d = ctx.upload(s.flat)
    v = base[:, :9].reshape(-1, 3)
    lo, hi = v.min(0).values, v.max(0).values
    g = torch.Generator(device="cuda:0").manual_seed(1)
    o = (lo + hi) / 2 + torch.randn(nrays, 3, device="cuda:0", generator=g) * float((hi - lo).max())
    tgt = lo + torch.rand(nrays, 3, device="cuda:0", generator=g) * (hi - lo)
    rays = torch.cat([o, (tgt - o) / (tgt - o).norm(dim=1, keepdim=True)], 1).contiguous()
    light = hi + (hi - lo)
    srays = torch.cat([o, (light - o) / (light - o).norm(dim=1, keepdim=True)], 1).contiguous()
    sdist = (light - o).norm(dim=1).contiguous()
    host_rays, host_srays = rays.cpu().numpy(), srays.cpu().numpy()
    step_ms = []
    try:
        for k in range(steps + 1):  # step 0: warm-up
            rec = twist_device(base, twist * max(k, 1) / steps)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with torch.cuda.stream(stream):
                d.mesh_update(rec, refit=refit)
                if device_queries:
                    d.query(rays)
                    d.query(srays, tmax=sdist, any_hit=True)
            if device_queries:
                stream.synchronize()
            else:
                d.intersect_rays(host_rays)
                d.intersect_rays(host_srays)
            if k:
                step_ms.append((time.perf_counter() - t0) * 1e3)
    finally:
        d.close()
    return dict(step_ms_sum=sum(step_ms), step_ms_median=float(np.median(step_ms)), step_ms=[round(x, 4) for x in step_ms])


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--sizes", default="4096,65536,1048576,16777216")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--twist", type=float, default=1.5)
    ap.add_argument("--step-rays", type=int, default=4096)
    a = ap.parse_args()
    ctx = rtb200.Context(0)
    stream = torch.cuda.Stream(device=0)
    res = dict(gpu=gpu_info(), workloads=[])
    tmp = tempfile.mkdtemp(prefix="ray_query_probe_")
    torus = os.path.join(tmp, "torus_1000000.stl")
    rtb200.write_stl(torus, rtb200.torus_triangles(1_000_000, seed=1_000_000))
    jobs = [("torus_1m_mesh", lambda: scene(True, torus)), ("ball_mesh", lambda: scene(True, None)),
            ("p5_sah", lambda: rtb200.PresetScene(5, "sah", 150))]
    for name, make in jobs:
        s = make()
        d = ctx.upload(s.flat)
        for n in [int(x) for x in a.sizes.split(",") if x]:
            entry = dict(workload=name, **measure(d, s.camera, n, stream, a.reps if n < (1 << 24) else 3))
            print(json.dumps(entry), flush=True)
            res["workloads"].append(entry)
        d.close()
        s.close()
    s = scene(True, torus)
    f = s.flat.contents
    base = torch.from_numpy(np.ctypeslib.as_array(f.loose_tri, shape=(f.n_loose, 12)).copy()).cuda()
    res["twist_sequence"] = dict(steps=a.steps, twist=a.twist, rays_per_step=a.step_rays, modes={})
    for mode in ("refit", "rebuild"):
        for q in ("device_query", "intersect_rays"):
            r = twist_sequence(ctx, s, base, a.twist, a.steps, a.step_rays, stream, mode == "refit", q == "device_query")
            res["twist_sequence"]["modes"][f"{mode}_{q}"] = r
            print(json.dumps({f"{mode}_{q}": {k: v for k, v in r.items() if k != "step_ms"}}), flush=True)
    s.close()
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
