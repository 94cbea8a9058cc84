"""In-place mesh updates (rtb_scene_mesh_update) against freeing the scene and uploading it again, on the GPU.

Workloads: preset 3 with its STL loaded as a mesh -- the 528-triangle ball, and seeded tori of about 10 k, 100 k and 1 M
triangles written as binary STL and loaded through the preset's STL path.  The new records are a growing twist of the model
about its vertical axis (tests/test_mesh_update.py: twist), computed by torch ops on the device.

  first uploads: the first 4 uploads of the scene into a new context (host clock to a device synchronisation).
  update:   refit and rebuild from device records (CUDA events on the caller's stream around the call, and a host clock to
            a device synchronisation), refit and rebuild from host records (host clock), and free + rtb_scene_upload of the
            same scene with the new records (host clock); the median of --reps, after a warm-up of each.
  sequence: a 30-step deformation, the twist growing from 0 to --twist (large motion) or --small-twist radians (small
            motion): each step updates the mesh from device records, then renders a Simple() 400x300 frame, or -- the large
            motion again -- intersects --rays rays from around the model (rtb_intersect_rays: a query workload, such as
            collision tests, whose cost per step is small next to an update).  Per mode (refit every step, rebuild every
            step, free + upload every step): update ms and consumer ms (frame kernel ms, or the query's host clock) per
            step, and the step's total (host clock, update + consumer).

The GPU name and power limit are read in the same call.

    python tools/mesh_update_probe.py --out profiles/r04_mesh_update_probe.json
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


def twist_device(base, amount):
    """[n][12] records (a, b, c, normal) twisted about the vertical axis through the model's centre by up to `amount` radians,
    growing with height; normals recomputed.  float32 torch ops on the device."""
    v = base[:, :9].reshape(-1, 3)
    lo, hi = v.min(0).values, v.max(0).values
    c = (lo + hi) / 2
    p = v - c
    a = amount * (v[:, 1] - lo[1]) / (hi[1] - lo[1])
    x = p[:, 0] * torch.cos(a) - p[:, 2] * torch.sin(a)
    z = p[:, 0] * torch.sin(a) + p[:, 2] * torch.cos(a)
    w = (torch.stack([x, p[:, 1], z], 1) + c).reshape(-1, 3, 3)
    n = torch.linalg.cross(w[:, 1] - w[:, 0], w[:, 2] - w[:, 0])
    n = n / n.norm(dim=1, keepdim=True).clamp_min(1e-30)
    return torch.cat([w.reshape(-1, 9), n], 1).contiguous()


def set_loose(s, records):
    f = s.flat.contents
    np.ctypeslib.as_array(f.loose_tri, shape=(f.n_loose * 12,))[:] = records.ravel()


def time_update(d, rec, refit, stream):
    """(event ms, host ms) of one update from `rec` (a CUDA tensor: events on `stream`; a numpy array: host clock only)."""
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    with torch.cuda.stream(stream):
        e0.record(stream)
        d.mesh_update(rec, refit=refit)
        e1.record(stream)
    torch.cuda.synchronize()
    host = (time.perf_counter() - t0) * 1e3
    return (e0.elapsed_time(e1) if torch.is_tensor(rec) else None), host


def time_reupload(ctx, d, s):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    d.close()
    d = ctx.upload(s.flat)
    torch.cuda.synchronize()
    return d, (time.perf_counter() - t0) * 1e3


def med(x):
    return float(np.median(x))


def first_uploads(s, n=4):
    """host ms of the first n uploads of the scene into a new context (each scene freed before the next): the first one
    also allocates the context's page-locked staging ring and grows the device memory pool."""
    c = rtb200.Context(0)
    ms = []
    try:
        for _ in range(n):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            d = c.upload(s.flat)
            torch.cuda.synchronize()
            ms.append((time.perf_counter() - t0) * 1e3)
            d.close()
    finally:
        c.close()
    return ms


def measure_updates(ctx, s, base, amount, reps, stream):
    new = twist_device(base, amount)
    new_host = new.cpu().numpy()
    d = ctx.upload(s.flat)
    out = {}
    try:
        for name, rec, refit in (("refit_device", new, True), ("rebuild_device", new, False),
                                 ("refit_host", new_host, True), ("rebuild_host", new_host, False)):
            time_update(d, rec, refit, stream)  # warm-up
            ev, host = zip(*[time_update(d, rec, refit, stream) for _ in range(reps)])
            out[name] = dict(host_ms=med(host)) if ev[0] is None else dict(event_ms=med(ev), host_ms=med(host))
        set_loose(s, new_host)
        d, _ = time_reupload(ctx, d, s)  # warm-up
        ms = []
        for _ in range(reps):
            d, t = time_reupload(ctx, d, s)
            ms.append(t)
        out["free_upload"] = dict(host_ms=med(ms), upload_bytes=d.upload_bytes)
    finally:
        d.close()
    return out


def sequence(ctx, s, base, twist, steps, mode, stream, consumer, rays):
    """A deformation of `steps` steps under one mode; every step: update (or free + upload), then the consumer -- a Simple()
    400x300 frame ("frame", kernel ms from the frame's events) or a batch of rays through rtb_intersect_rays ("rays",
    host clock)."""
    set_loose(s, base.cpu().numpy())
    d = ctx.upload(s.flat)
    setting, frame = rtb200.make_setting("simple"), rtb200.make_frame(400, 300, seed=1)

    def consume():
        if consumer == "frame":
            return d.render(s.camera, setting, frame)[1]["kernel_ms"]
        t = time.perf_counter()
        d.intersect_rays(rays)
        return (time.perf_counter() - t) * 1e3

    consume()  # warm-up (a frame: the schedule of the view)
    upd, kern, total = [], [], []
    try:
        for k in range(1, steps + 1):
            rec = twist_device(base, twist * k / steps)
            if mode == "free_upload":
                set_loose(s, rec.cpu().numpy())
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if mode == "free_upload":
                d.close()
                d = ctx.upload(s.flat)
            else:
                with torch.cuda.stream(stream):
                    d.mesh_update(rec, refit=mode == "refit")
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            k_ms = consume()
            t2 = time.perf_counter()
            upd.append((t1 - t0) * 1e3)
            kern.append(k_ms)
            total.append((t2 - t0) * 1e3)
    finally:
        d.close()
    return dict(update_ms=[round(x, 4) for x in upd], consumer_ms=[round(x, 4) for x in kern],
                step_ms=[round(x, 4) for x in total], update_ms_sum=sum(upd), consumer_ms_sum=sum(kern),
                step_ms_sum=sum(total), consumer_ms_first=kern[0], consumer_ms_last=kern[-1])


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--twist", type=float, default=1.5, help="twist of the last step, radians")
    ap.add_argument("--small-twist", type=float, default=0.1, help="twist of the last step of the small-motion sequence")
    ap.add_argument("--rays", type=int, default=4096, help="rays per step of the ray-query sequence")
    ap.add_argument("--sizes", default="10000,100000,1000000")
    a = ap.parse_args()
    ctx = rtb200.Context(0)
    stream = torch.cuda.Stream(device=0)
    res = dict(gpu=gpu_info(), steps=a.steps, twist=a.twist, workloads=[])
    tmp = tempfile.mkdtemp(prefix="mesh_update_probe_")
    jobs = [("ball", None)]
    for n in [int(x) for x in a.sizes.split(",") if x]:
        path = os.path.join(tmp, f"torus_{n}.stl")
        rtb200.write_stl(path, rtb200.torus_triangles(n, seed=n))
        jobs.append((f"torus_{n}", path))
    for name, stl in jobs:
        s = scene(True, stl)
        f = s.flat.contents
        base_host = np.ctypeslib.as_array(f.loose_tri, shape=(f.n_loose, 12)).copy()
        base = torch.from_numpy(base_host).cuda()
        entry = dict(workload=name, triangles=int(f.n_loose))
        entry["first_uploads"] = first_uploads(s)
        entry["update"] = measure_updates(ctx, s, base, a.twist / 2, a.reps, stream)
        rng = np.random.default_rng(1)
        v = base_host[:, :9].reshape(-1, 3)
        lo, hi = v.min(0), v.max(0)
        o = (lo + hi) / 2 + rng.normal(size=(a.rays, 3)) * float(np.max(hi - lo))
        tgt = lo + rng.uniform(size=(a.rays, 3)) * (hi - lo)
        dirs = (tgt - o) / np.linalg.norm(tgt - o, axis=1, keepdims=True)
        rays = np.concatenate([o, dirs], 1).astype(np.float32)
        entry["sequence"] = {}
        for label, twist, consumer in (("frame_large_twist", a.twist, "frame"), ("frame_small_twist", a.small_twist, "frame"),
                                       ("rays_large_twist", a.twist, "rays")):
            entry["sequence"][label] = dict(twist=twist, consumer=consumer, modes={
                mode: sequence(ctx, s, base, twist, a.steps, mode, stream, consumer, rays) for mode in ("refit", "rebuild", "free_upload")})
        s.close()
        short = {k: v for k, v in entry.items() if k != "sequence"}
        short["sequence"] = {lab: {m: {k: v for k, v in r.items() if not isinstance(v, list)} for m, r in q["modes"].items()}
                             for lab, q in entry["sequence"].items()}
        print(json.dumps(short), flush=True)
        res["workloads"].append(entry)
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
