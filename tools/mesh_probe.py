"""Triangle meshes (RTB_PRIM_MESH) against the run of loose triangles with the same records, on the GPU.

Workloads: preset 3 (the 528-triangle STL ball in the smallpt box) at bench.py's p3_stl_64 configuration (400x300, Monte
Carlo Default(), 64 spp) and under Simple() (Whitted ray tree); seeded tori of about 10 k, 100 k and 1 M triangles written as
binary STL and loaded through the preset's STL path, rendered under Simple() at 400x300.  For each: Mrays/s and kernel ms,
triangle tests and nodes per ray (a separate counting render), upload + build ms (host clock from a device synchronisation
to the next, after one warm-up upload) and device bytes, and whether the run and
mesh images are bit-identical (the run is skipped above --run-max triangles).  The GPU name and power limit are read in the
same call.

    python tools/mesh_probe.py --out profiles/r03_mesh_probe.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rtb200  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # the measurement itself still needs the GPU; this is only the label
        return f"unknown ({e})"


def scene(mesh, stl):
    rtb200.set_stl_as_mesh(mesh)
    try:
        return rtb200.PresetScene(3, stl_path=stl)
    finally:
        rtb200.set_stl_as_mesh(False)


def timed_upload(ctx, flat):
    """rtb_scene_upload (copies + device builds are asynchronous) up to a device synchronisation, in ms."""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    d = ctx.upload(flat)
    torch.cuda.synchronize()
    return d, (time.perf_counter() - t0) * 1e3


def measure(ctx, mesh, stl, setting, w, h, spp, reps):
    s = scene(mesh, stl)
    timed_upload(ctx, s.flat)[0].close()  # warm-up: module loading, allocator pools
    d, upload_ms = timed_upload(ctx, s.flat)
    st = setting if setting is not None else s.setting
    try:
        frame = rtb200.make_frame(w, h, samples=spp, seed=1)
        img, stats = d.render(s.camera, st, frame)  # warm-up
        ks = []
        for _ in range(reps):
            img, stats = d.render(s.camera, st, frame)
            ks.append(stats["kernel_ms"])
        _, cst = d.render(s.camera, st, rtb200.make_frame(w, h, samples=spp, seed=1, counters=1))
        kms = float(np.median(ks))
        return img, dict(kernel_ms=kms, kernel_ms_min=float(np.min(ks)), n_rays=int(stats["n_rays"]),
                         mrays_per_s=stats["n_rays"] / kms / 1e3, tests_per_ray=cst["n_tri_tests"] / cst["n_rays"],
                         nodes_per_ray=cst["n_steps"] / cst["n_rays"], upload_build_ms=upload_ms,
                         device_bytes=d.device_bytes, upload_bytes=d.upload_bytes)
    finally:
        d.close()
        s.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--run-max", type=int, default=100_000, help="largest torus also rendered as a run")
    ap.add_argument("--sizes", default="10000,100000,1000000")
    a = ap.parse_args()
    ctx = rtb200.Context(0)
    res = dict(gpu=gpu_info(), workloads=[])
    tmp = tempfile.mkdtemp(prefix="mesh_probe_")
    jobs = [("p3_stl_64", None, None, 400, 300, 64), ("p3_simple", None, rtb200.make_setting("simple"), 400, 300, 1)]
    for n in [int(x) for x in a.sizes.split(",") if x]:
        path = os.path.join(tmp, f"torus_{n}.stl")
        rtb200.write_stl(path, rtb200.torus_triangles(n, seed=n))
        jobs.append((f"torus_{n}_simple", path, rtb200.make_setting("simple"), 400, 300, 1))
    for name, stl, setting, w, h, spp in jobs:
        entry = dict(workload=name, width=w, height=h, spp=spp)
        n_tris = None
        img_m, entry["mesh"] = measure(ctx, True, stl, setting, w, h, spp, a.reps)
        s = scene(True, stl)
        n_tris = s.flat.contents.n_loose
        s.close()
        entry["triangles"] = n_tris
        if n_tris <= a.run_max:
            img_r, entry["run"] = measure(ctx, False, stl, setting, w, h, spp, a.reps)
            entry["bit_identical"] = img_r.tobytes() == img_m.tobytes()
            entry["speedup"] = entry["run"]["kernel_ms"] / entry["mesh"]["kernel_ms"]
        print(json.dumps(entry), flush=True)
        res["workloads"].append(entry)
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
