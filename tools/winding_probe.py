"""Winding-number queries on device buffers (rtb_query_winding), on the GPU.

Scenes: seeded tori (rtb200.torus_triangles with two vertices swapped so that the facets face outwards, tube radius 6) of
10 k, 100 k and 1 M triangles as a MESH record.  Point sets, made by torch ops on the device (point_query_probe.point_sets):
near the surface (up to +-1 % of the tube radius along the normal, in triangle order), the same shuffled, and uniform in the
model's box.

Measured, CUDA-event ms of one call on a side stream with preallocated outputs, the median of --reps after a warm-up:
  * moments: rtb_scene_mesh_moments on a fresh upload of each torus (each call on a new scene: the call builds once);
  * winding_numbers on 1 Mi and 16 Mi points of each set at beta 2 and 4, and beta = inf (exact) on the 10 k torus only;
  * signed_distance end to end (closest_points + winding + torch's elementwise ops) next to closest_points alone on the same
    points;
  * the 30-step refit twist of the 1 M torus (mesh_update_probe.twist_device), each step a refit from device records
    followed by 64 Ki containment queries on the same stream, one synchronise per step; host clock per step, summed.
The 16 Mi inputs and outputs (256 MB) do not fit the 126 MB L2.  The GPU name, power limit and max SM clock are read in the
same call.

    python tools/winding_probe.py --out profiles/r07_winding_probe.json
"""
import argparse
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
from point_query_probe import flat_scene, point_sets  # noqa: E402
from ray_query_probe import event_ms  # noqa: E402


def torus(n):
    f = rtb200.torus_triangles(n, seed=n)
    return np.concatenate([f[:, 3:6], f[:, 9:12], f[:, 6:9], -f[:, :3]], 1).astype(np.float32)


def moments_ms(ctx, tris, stream, reps):
    ms = []
    for _ in range(reps + 1):  # the first: warm-up
        d = ctx.upload(flat_scene(tris, rtb200.PRIM_MESH))
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        d.mesh_moments(stream=stream.cuda_stream)
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
        d.close()
    return float(np.median(ms[1:]))


def measure(d, tris, n, stream, reps, betas):
    sets = point_sets(tris, n, 6.0, n)
    w = torch.empty(n, device="cuda:0")
    torch.cuda.synchronize()  # the points are made on the default stream, the queries run on `stream`
    res = dict(points=n)
    for kind, pts in sets.items():
        e = dict()
        for beta in betas:
            e[f"winding_beta{beta}_ms"] = event_ms(lambda: d.winding_numbers(pts, beta=beta, stream=stream.cuda_stream, out=w), stream, reps)
            e[f"inside_fraction_beta{beta}"] = float((w > 0.5).float().mean())
        res[kind] = e
    return res


def signed_distance(d, tris, n, stream, reps):
    pts = point_sets(tris, n, 6.0, n + 1)["near"]
    out_c = (torch.empty(n, dtype=torch.int32, device="cuda:0"), torch.empty(n, device="cuda:0"),
             torch.empty(n, 3, device="cuda:0"), torch.empty(n, 3, device="cuda:0"))
    torch.cuda.synchronize()
    return dict(points=n, closest_points_ms=event_ms(lambda: d.closest_points(pts, out=out_c, stream=stream.cuda_stream), stream, reps),
                signed_distance_ms=event_ms(lambda: d.signed_distance(pts, stream=stream.cuda_stream), stream, reps))


def twist_sequence(ctx, tris, steps, twist, npts, stream):
    d = ctx.upload(flat_scene(tris, rtb200.PRIM_MESH))
    base = torch.from_numpy(tris).cuda()
    pts = point_sets(tris, npts, 6.0, 1)["near"]
    out = torch.empty(npts, dtype=torch.bool, device="cuda:0")
    torch.cuda.synchronize()
    step_ms = []
    try:
        d.mesh_moments()
        for k in range(steps + 1):  # step 0: warm-up
            rec = twist_device(base, twist * max(k, 1) / steps)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with torch.cuda.stream(stream):
                d.mesh_update(rec, refit=True)
                d.contains(pts, out=out)
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
    ap.add_argument("--sizes", default="1048576,16777216")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--twist", type=float, default=1.5)
    ap.add_argument("--step-points", type=int, default=65536)
    a = ap.parse_args()
    ctx = rtb200.Context(0)
    stream = torch.cuda.Stream(device=0)
    res = dict(gpu=gpu_info(), moments=[], workloads=[], signed_distance=[])
    for n_tris in (10_000, 100_000, 1_000_000):
        tris = torus(n_tris)
        entry = dict(workload=f"torus_{n_tris // 1000}k_mesh" if n_tris < 1_000_000 else "torus_1m_mesh", triangles=len(tris),
                     moments_ms=moments_ms(ctx, tris, stream, a.reps))
        print(json.dumps(entry), flush=True)
        res["moments"].append(entry)
        d = ctx.upload(flat_scene(tris, rtb200.PRIM_MESH))
        d.mesh_moments()
        for n in [int(x) for x in a.sizes.split(",") if x]:
            betas = [2.0, 4.0] + ([float("inf")] if n_tris == 10_000 else [])
            e = dict(workload=entry["workload"], triangles=len(tris), **measure(d, tris, n, stream, a.reps if n < (1 << 24) else 3, betas))
            print(json.dumps(e), flush=True)
            res["workloads"].append(e)
            e = dict(workload=entry["workload"], **signed_distance(d, tris, n, stream, a.reps if n < (1 << 24) else 3))
            print(json.dumps(e), flush=True)
            res["signed_distance"].append(e)
        d.close()
    r = twist_sequence(ctx, torus(1_000_000), a.steps, a.twist, a.step_points, stream)
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
