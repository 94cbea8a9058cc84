"""Triangle intersection queries on device buffers (rtb_query_triangles), on the GPU.

Scene: a seeded torus of 1 M triangles (rtb200.torus_triangles, major radius 15, tube radius 6) as a MESH record.  Query sets:
a second torus of 10 k, 100 k and 1 M triangles, placed three ways:
  * interpenetrating: rotated by 0.5 rad about the x axis and shifted by (2, 0.5, 1), so that much of its surface crosses;
  * touching: shifted by 42 along x (twice the outer radius), so that the tubes meet near one place and the boxes of the
    triangles there overlap;
  * far: shifted by 1000 along x.
Measured, CUDA-event ms of one call on a side stream with preallocated outputs, the median of --reps after a warm-up:
  * intersects (RTB_QUERY_ANY) and the PAIRS mode (a raw call with a buffer of 4 m pairs and the count on the device, no
    read-back), with the number of pairs;
  * the 10 k torus as a TRIANGLES run (every query triangle against every triangle) next to the same torus as a mesh: the
    brute-force baseline;
  * a 30-step refit twist of the 1 M torus (mesh_update_probe.twist_device), each step a refit from device records followed by
    intersects on 64 Ki interpenetrating query triangles on the same stream, one synchronise per step; host clock per step.
  * the fraction of leaf tests (query and scene triangle with overlapping boxes) that took an exact fallback, counted with the
    host build of csrc/rtb_tritri.h on a sample of 2,000 query triangles of each placement against the 1 M torus.
The GPU name, power limit and max SM clock are read in the same call.

    python tools/triangle_query_probe.py --out profiles/r08_triangle_query_probe.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rtb200  # noqa: E402
from mesh_probe import gpu_info  # noqa: E402
from mesh_update_probe import twist_device  # noqa: E402
from point_query_probe import flat_scene  # noqa: E402
from ray_query_probe import event_ms  # noqa: E402


def torus(n, seed):
    f = rtb200.torus_triangles(n, seed=seed)
    return np.ascontiguousarray(np.concatenate([f[:, 3:12], f[:, :3]], 1), np.float32)


def placed(tris, how):
    v = tris[:, :9].reshape(-1, 3).astype(np.float64)
    if how == "interpenetrating":
        v = v - (0.0, 16.0, 0.0)
        c, s = np.cos(0.5), np.sin(0.5)
        v = np.stack([v[:, 0], c * v[:, 1] - s * v[:, 2], s * v[:, 1] + c * v[:, 2]], 1) + (0.0, 16.0, 0.0) + (2.0, 0.5, 1.0)
    else:
        v = v + ((42.0 if how == "touching" else 1000.0), 0.0, 0.0)
    out = tris.copy()
    out[:, :9] = v.reshape(-1, 9).astype(np.float32)
    return out


def pairs_call(ctx, d, q, buf, count, stream):
    rc = ctx._lib.rtb_query_triangles(ctx._h, d._h, q.shape[0], C.c_void_p(q.data_ptr()), rtb200.QUERY_PAIRS, None,
                                      C.c_void_p(buf.data_ptr()), buf.shape[0], C.c_void_p(count.data_ptr()),
                                      C.c_void_p(stream.cuda_stream))
    assert rc == 0, rc


def measure(ctx, d, queries, stream, reps):
    q = torch.from_numpy(queries).cuda()
    m = q.shape[0]
    hit = torch.empty(m, dtype=torch.bool, device="cuda:0")
    buf = torch.empty((4 * m, 2), dtype=torch.int32, device="cuda:0")
    count = torch.empty(1, dtype=torch.int64, device="cuda:0")
    torch.cuda.synchronize()
    any_ms = event_ms(lambda: d.intersects(q, stream=stream.cuda_stream, out=hit), stream, reps)
    pairs_ms = event_ms(lambda: pairs_call(ctx, d, q, buf, count, stream), stream, reps)
    return dict(query_triangles=m, any_ms=any_ms, pairs_ms=pairs_ms, pairs=int(count.item()), intersecting=int(hit.sum()))


_HOST_SRC = r"""
static long g_exact;
#define RTB_TRITRI_COUNT(k) (++g_exact)
#include "rtb_tritri.h"
// leaf tests (box-overlapping pairs) of the query triangles q[n][12] against t[m][12] (a, b, c, n), and how many of them ran
// at least one exact evaluation
extern "C" void leaf_tests(const float *q, long n, const float *t, long m, long *tests, long *fell, long *hits)
{
    *tests = *fell = *hits = 0;
    for (long i = 0; i < n; i++)
    {
        const float *p = q + 12 * i;
        if (rtb_tritri::degenerate(p)) continue;
        float lo[3], hi[3], tlo[3], thi[3];
        rtb_tritri::box(p, lo, hi);
        for (long k = 0; k < m; k++)
        {
            const float *v = t + 12 * k;
            rtb_tritri::box(v, tlo, thi);
            if (!rtb_tritri::boxesOverlap(lo, hi, tlo, thi)) continue;
            const long e = g_exact;
            *hits += rtb_tritri::meets(p, v);
            ++*tests;
            *fell += g_exact != e;
        }
    }
}
"""


def fallback_fraction(tris, sample):
    d = tempfile.mkdtemp()
    src, so = os.path.join(d, "h.cpp"), os.path.join(d, "h.so")
    open(src, "w").write(_HOST_SRC)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-I",
                           os.path.join(rtb200.PKG, "csrc"), "-o", so, src])
    lib = C.CDLL(so)
    lib.leaf_tests.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_long] + [C.POINTER(C.c_long)] * 3
    # the scene's triangles as the query sees them: (a, fl(a - e1), fl(a - e2))
    a = tris[:, 0:3]
    e1, e2 = (a - tris[:, 3:6]).astype(np.float32), (a - tris[:, 6:9]).astype(np.float32)
    t = np.ascontiguousarray(np.concatenate([a, a - e1, a - e2, tris[:, 9:12]], 1), np.float32)
    out = {}
    for how, q in sample.items():
        q = np.ascontiguousarray(q, np.float32)
        tests, fell, hits = C.c_long(), C.c_long(), C.c_long()
        lib.leaf_tests(q.ctypes.data, len(q), t.ctypes.data, len(t), C.byref(tests), C.byref(fell), C.byref(hits))
        out[how] = dict(query_triangles=len(q), leaf_tests=tests.value, exact_fallback=fell.value, intersecting_pairs=hits.value,
                        fallback_fraction=fell.value / max(tests.value, 1))
    return out


def twist_sequence(ctx, tris, steps, twist, nq, stream):
    d = ctx.upload(flat_scene(tris, rtb200.PRIM_MESH))
    base = torch.from_numpy(tris).cuda()
    q = torch.from_numpy(placed(torus(nq, 3), "interpenetrating")).cuda()
    out = torch.empty(nq, dtype=torch.bool, device="cuda:0")
    torch.cuda.synchronize()
    step_ms = []
    try:
        for k in range(steps + 1):  # step 0: warm-up
            rec = twist_device(base, twist * max(k, 1) / steps)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with torch.cuda.stream(stream):
                d.mesh_update(rec, refit=True)
                d.intersects(q, out=out)
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
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--twist", type=float, default=1.5)
    ap.add_argument("--step-triangles", type=int, default=65536)
    ap.add_argument("--sample", type=int, default=2000)
    a = ap.parse_args()
    ctx = rtb200.Context(0)
    stream = torch.cuda.Stream(device=0)
    res = dict(gpu=gpu_info(), workloads=[])
    big = torus(1_000_000, 1)
    d = ctx.upload(flat_scene(big, rtb200.PRIM_MESH))
    for n in (10_000, 100_000, 1_000_000):
        for how in ("interpenetrating", "touching", "far"):
            e = dict(workload=f"torus_1m_mesh vs {how} torus of {n}", **measure(ctx, d, placed(torus(n, 2), how), stream, a.reps))
            print(json.dumps(e), flush=True)
            res["workloads"].append(e)
    d.close()
    small, q = torus(10_000, 1), placed(torus(10_000, 2), "interpenetrating")
    for prim, name in ((rtb200.PRIM_TRIANGLES, "run"), (rtb200.PRIM_MESH, "mesh")):
        d = ctx.upload(flat_scene(small, prim))
        e = dict(workload=f"torus_10k_{name} vs interpenetrating torus of 10000", **measure(ctx, d, q, stream, a.reps))
        print(json.dumps(e), flush=True)
        res["workloads"].append(e)
        d.close()
    r = twist_sequence(ctx, big, a.steps, a.twist, a.step_triangles, stream)
    res["twist_sequence"] = dict(steps=a.steps, twist=a.twist, query_triangles_per_step=a.step_triangles, mode="refit", **r)
    print(json.dumps({k: v for k, v in res["twist_sequence"].items() if k != "step_ms"}), flush=True)
    ctx.close()
    rng = np.random.default_rng(4)
    sample = {how: placed(torus(1_000_000, 2), how)[rng.choice(1_000_000, a.sample, replace=False)]
              for how in ("interpenetrating", "touching")}
    res["exact_fallback_host"] = fallback_fraction(big, sample)
    print(json.dumps(res["exact_fallback_host"]), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
