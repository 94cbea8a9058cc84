#!/usr/bin/env python
"""bench.py -- Mrays/s of the ray-generation / intersection / shading hot path on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--gather peer|nccl]
                  [--dump-outputs DIR]
  (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

--dump-outputs DIR writes what the last timed step computed as .npy files: the frame (a fixed sample of 2 Mi pixels of a
larger frame), or for pt_r2000_150 every accelerator's per-ray results.  Two builds run with the same arguments get the
same seeded inputs and can be compared output for output.

A step = one frame of the workload rendered by the hot path (ray generation -> accelerator traversal -> triangle /
sphere / plane tests -> Whitted or Monte-Carlo shading -> framebuffer).  For N > 1 the frame is sharded over the ranks
(tile rows up to 4 ranks, column blocks above) and every rank stores its tiles straight into rank 0's frame over NVLink
(CUDA IPC mapping, RTB_LAYOUT_GLOBAL); a one-word NCCL all-reduce closes the step (`--gather nccl`: the round-1 path,
all_gather_into_tensor + unshard kernel).

  value      the frame with the scene resident in HBM, timed with CUDA events on the launching stream, max over ranks.
             STEADY STATE of one view: from the second frame of a view on the library renders its tiles heaviest first
             and gives the latency-critical ones to its latency tiers; `first_frame_ms` (fresh schedule, raster order)
             and `moving_camera_ms` (order kept, tiers off) are reported next to it.
  e2e        the same frame through the reference-facing host-buffer calls, every step: scene upload (H2D) +
             render + the assembled float frame in ONE page-locked host buffer (N = 1: rtb_scene_upload + rtb_render;
             N > 1: rank 0's host thread drives all N devices through rtb_multi_*).
  roofline   warp-instruction issue: instructions of the frame (ncu of HEAD, profiles/r02_issue_counts.json) / (SMs x 4
             schedulers x SM clock observed during the run x kernel time measured by this run).
  cpu_baseline / --impl reference: the reference's own Render() (oracle/_ref, else the port) on the host cores, on the
             SAME frame (width, height, spp); the N = 1 line also checks the GPU frame against it (`parity_checked`).

Prints ONE JSON line (rank 0).
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json: "150-segment tunnel (k-d tree SAH ...)", config[4] "4K tunnel ... stress render"
    "p5_sah_4k": dict(preset=5, algorithm="sah", segments=150, width=3840, height=2880, samples=1,
                      desc="preset 5 long narrow tunnel, 150-segment tessellation (45,900 triangles), k-d tree SAH "
                           "(leaf<=8, depth<=18), Whitted Simple() maxDepth 20, 3840x2880 (4:3), 1 spp"),
    "p5_rgrid_4k": dict(preset=5, algorithm="rgrid", segments=150, width=3840, height=2880, samples=1,
                        desc="preset 5, regular grid 400x5x400, Whitted Simple(), 3840x2880, 1 spp"),
    "p5_kd_4k": dict(preset=5, algorithm="kd", segments=150, width=3840, height=2880, samples=1,
                     desc="preset 5, k-d median, Whitted, 3840x2880, 1 spp"),
    "p5_fgrid_4k": dict(preset=5, algorithm="fgrid", segments=150, width=3840, height=2880, samples=1,
                        desc="preset 5, flat grid 400^3, Whitted, 3840x2880, 1 spp"),
    "p4_sah_4k": dict(preset=4, algorithm="sah", segments=150, width=3840, height=2880, samples=1,
                      desc="preset 4 short wide tunnel, k-d SAH, Whitted, 3840x2880, 1 spp"),
    "p4_rgrid_4k": dict(preset=4, algorithm="rgrid", segments=150, width=3840, height=2880, samples=1,
                        desc="preset 4 short wide tunnel, regular grid 350x166x400, Whitted, 3840x2880, 1 spp"),
    "p2_smallpt_64": dict(preset=2, algorithm="linear", segments=0, width=1280, height=960, samples=64,
                          desc="preset 2 smallpt Cornell box, Monte Carlo Default(), 1280x960, 64 spp"),
    "p2_smallpt_256": dict(preset=2, algorithm="linear", segments=0, width=400, height=300, samples=256,
                           desc="preset 2 smallpt, Monte Carlo Default(), demo default 400x300, 256 spp"),
    "p2_smallpt_1024": dict(preset=2, algorithm="linear", segments=0, width=400, height=300, samples=1024,
                            desc="preset 2 smallpt, Monte Carlo Default(), demo default 400x300, 1024 spp"),
    "p3_stl_64": dict(preset=3, algorithm="linear", segments=0, width=400, height=300, samples=64,
                      desc="preset 3 smallpt with the 528-triangle STL ball (no accelerator), Monte Carlo Default(), 400x300, 64 spp"),
    "p1_mc_64": dict(preset=1, algorithm="linear", segments=0, width=1280, height=960, samples=64,
                     desc="preset 1 emissive checker ground + two diffuse spheres, Monte Carlo Default(), 1280x960, 64 spp"),
    "p1_simple_4k": dict(preset=1, algorithm="linear", segments=0, width=3840, height=2880, samples=1, setting="simple",
                         desc="preset 1 under Simple() (BASELINE config[0]'s 'Whitted, 1 spp' wording), 3840x2880"),
    "p5_sah_400": dict(preset=5, algorithm="sah", segments=150, width=400, height=300, samples=1,
                       desc="preset 5, k-d SAH, Whitted, demo default 400x300, 1 spp"),
    "p5_rgrid_400": dict(preset=5, algorithm="rgrid", segments=150, width=400, height=300, samples=1,
                         desc="preset 5, regular grid 400x5x400, Whitted, demo default 400x300, 1 spp"),
    "p4_rgrid_400": dict(preset=4, algorithm="rgrid", segments=150, width=400, height=300, samples=1,
                         desc="preset 4, regular grid 350x166x400, Whitted, demo default 400x300, 1 spp"),
    # the reference's PerformanceTest console program (PT/main.cpp:127-173): BASELINE.md's last table
    "pt_r2000_150": dict(kind="pt", radius=2000.0, angle=1.5708, arch_seg=150, path_seg=150, rays=1000,
                         desc="PerformanceTest: tunnel radius 2000, 150 x 150 segments, 1000 random rays, <= 200 mirror bounces to the exit plane"),
}
EXTRAS = ["p5_rgrid_4k", "p5_kd_4k", "p5_fgrid_4k", "p4_sah_4k", "p4_rgrid_4k", "p2_smallpt_64", "p1_mc_64", "p3_stl_64",
          "p5_sah_400", "p5_rgrid_400"]
ROW_BLOCK = int(os.environ.get("RTB_ROW_BLOCK", "8"))  # rows per dealt block (multiple of 8)
# N > 1: column-block shards (rtb_frame.col_block) -- every rank renders every row and 1 / N of the 32-pixel column
# blocks, so all ranks hold the same mix of heavy (vanishing point) and light tiles; 0 = whole-row shards
COL_BLOCK = int(os.environ.get("RTB_COL_BLOCK", "32"))
# ... from this many ranks on: up to 4 ranks the few heavy row blocks around the vanishing point already land on
# different ranks (measured: N = 2 rows 10,054 vs columns 9,833 Mrays/s); at 8 ranks rows leave half the ranks without them
COL_MIN_WORLD = int(os.environ.get("RTB_COL_MIN_WORLD", "5"))
METRIC = "Mrays/s on tunnel scenes (grid/k-d tree) at 1/2/4/8 B200 vs CPU render secs"
N_SM, SCHEDULERS = 148, 4


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback (B200_PROFILING.md)"


def issue_counts(wl_name):
    """Warp instructions of one steady-state frame of the workload, per kernel, from the ncu capture of HEAD's kernels
    (profiles/r02_issue_counts.json, written by profiles/r02_collect.py from `ncu --set full`)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_issue_counts.json")) as f:
            prof = json.load(f)
        return prof["workloads"].get(wl_name), prof.get("source")
    except Exception:
        return None, None


# ---- clocks: sampled while the timed region runs ----------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def start(self):
        if self._nv:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join()
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---- the reference arm / cpu baseline ----------------------------------------------------------------
def cpu_reference(wl, repeat, warmup=0, image=False):
    """The reference's own Render() on the host cores (all threads), on the workload's own frame.
    Timing comes from the hooks-free build (ref_timing); the ray count -- and, with image=True, the frame the GPU result
    is checked against -- from the build with the counting hooks (ref), else from the port (oracle)."""
    from oracle import oracle_py as O
    kind = "reference" if O.available("ref_timing") else "port"
    which = "ref_timing" if kind == "reference" else "oracle"
    cores = os.cpu_count() or 1
    kw = dict(preset=wl["preset"], algorithm=wl["algorithm"], segments=wl["segments"], width=wl["width"], height=wl["height"],
              samples=wl["samples"], threads=cores, setting=wl.get("setting", "preset"))
    counted = O.run("ref" if O.available("ref") else "oracle", repeat=1, image=image, **kw)
    r = O.run(which, repeat=repeat + warmup, **kw)
    times = np.asarray(r["render_ms_all"][warmup:], np.float64)
    return dict(kind=kind, cores=cores, rays=int(counted["n_rays"]), ms=times, prepare_ms=float(r["prepare_ms"]),
                image=counted.get("image"))


def cpu_repeats(wl, budget_s=30.0):
    """How many Render() calls of this workload fit the CPU budget (estimated from the survey's per-core rates)."""
    cores = os.cpu_count() or 1
    samples = wl["width"] * wl["height"] * wl["samples"]
    rays_per_sample = {1: 2.0, 2: 8.3, 3: 8.4, 4: 2.1, 5: 3.1}[wl["preset"]] if wl.get("setting") != "simple" else 1.5
    rate = {1: 3.4e6, 2: 2.0e6, 3: 0.055e6, 4: 0.4e6, 5: 0.9e6}[wl["preset"]] * cores * 0.8  # rays / s
    est = samples * rays_per_sample / rate
    return max(1, min(5, int(budget_s / max(est, 1e-3)))), est


_JSON_FD = None


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


DUMP_PIXELS = 1 << 21  # 2 Mi pixels: 24 MiB of float32 RGB + 16 MiB of float64 pixel indices


def dump_outputs(out_dir, arrays, image=None):
    """--dump-outputs: every array of `arrays` as out_dir/<name>.npy (float32 stays float32, anything else becomes
    float64), and the frame `image` [H][W][3] float32 as image.npy.  A frame of more than DUMP_PIXELS pixels is
    written as a fixed sample (seed 0) of that many pixels, [n][3], with their flat indices y * W + x, ascending,
    as image_pixels.npy -- the same pixels for every run of the same frame size."""
    os.makedirs(out_dir, exist_ok=True)
    out = dict(arrays)
    if image is not None:
        flat = np.ascontiguousarray(image, np.float32).reshape(-1, image.shape[-1])
        if flat.shape[0] > DUMP_PIXELS:
            idx = np.sort(np.random.default_rng(0).choice(flat.shape[0], DUMP_PIXELS, replace=False))
            out["image"], out["image_pixels"] = flat[idx], idx
        else:
            out["image"] = image
    for name, a in out.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float32 if a.dtype == np.float32 else np.float64))


def run_reference(args, wl_name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[wl_name]
    if wl.get("kind") == "pt":
        return run_pt_reference(args, wl_name)
    # the SAME frame as the B200 arm: width, height, spp, setting.  A 4K tunnel frame is ~2-4 s of Render() on a 16-core
    # host; Monte-Carlo frames cost more, so the number of timed Render() calls is bounded (stated in `sample`).
    fit, est = cpu_repeats(wl, budget_s=150.0)
    steps = min(args.steps, max(fit, 1)) if wl["samples"] > 1 else args.steps
    warm = min(args.warmup, 1) if wl["samples"] > 1 else args.warmup
    res = cpu_reference(wl, steps, warm)
    ms = float(res["ms"].mean())
    value = res["rays"] / ms / 1e3
    sample = f"the whole {wl['width']}x{wl['height']} frame at {wl['samples']} spp, {steps} timed Render() call(s) after {warm} warm-up"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "same_config": True,
            "config": {"workload": wl_name, "description": wl["desc"], "sample": sample, "rays_per_step": res["rays"]},
            "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": res["cores"], "kind": res["kind"], "sample": sample,
                             "render_s": ms / 1e3, "prepare_s": res["prepare_ms"] / 1e3},
            "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ---- PerformanceTest workload (BASELINE.md last table) ---------------------------------------------------------------
PT_PUBLISHED_TRACE_MS = {"rgrid": 292.0, "fgrid": 1213.8, "kd": 644.3, "sah": 223.3, "convex": 134.3}  # 2000, 150, 150 (len-*.log)
PT_ALGS = ["rgrid", "fgrid", "kd", "sah", "convex"]


def pt_rays(n, seed=5):
    return np.random.default_rng(seed).random((n, 2), dtype=np.float32)


def run_pt_reference(args, wl_name):
    from oracle import oracle_py as O
    wl = WORKLOADS[wl_name]
    xy = pt_rays(wl["rays"])
    which = "ref_pt" if O.available("ref_pt") else "oracle"
    table = {}
    for alg in PT_ALGS:
        if which == "oracle" and alg == "convex":
            continue
        t = []
        for _ in range(max(1, min(args.steps, 3))):
            r = O.bounce(which, xy, wl["radius"], wl["angle"], wl["arch_seg"], wl["path_seg"], alg, 200, threads=1, pt_builders=True)
            t.append(r["trace_ms"])
        table[alg] = {"trace_ms": float(np.mean(t)), "prepare_ms": r["prepare_ms"], "total_rays": int(r["total_rays"])}
    v = table["sah"]["trace_ms"]
    sample = f"{wl['rays']} rays, single thread as the reference program runs it, {max(1, min(args.steps, 3))} run(s) per accelerator"
    emit({"impl": "reference", "metric": "PerformanceTest trace ms (k-d SAH; 1000 random rays, <= 200 mirror bounces)", "value": v, "unit": "ms",
          "n_gpus": args.gpus, "steps": max(1, min(args.steps, 3)), "warmup": 0, "ms_per_step": v, "higher_is_better": False, "scaling": "strong",
          "vs_baseline": v / PT_PUBLISHED_TRACE_MS["sah"], "dtype": "f32", "data": "synthetic",
          "config": {"workload": wl_name, "description": wl["desc"], "table": table, "published_trace_ms": PT_PUBLISHED_TRACE_MS},
          "cpu_baseline": {"value": v, "unit": "ms", "cores": 1, "kind": "reference" if which == "ref_pt" else "port", "sample": sample},
          "e2e": {"value": v, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0})


def run_pt(args, wl_name):
    """rt::PerformanceTest (host/rt_render.cpp) -> rtb_bounce_rays: the reference program's ray loop on the GPU."""
    import rtb200
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[wl_name]
    xy = pt_rays(wl["rays"])
    big = pt_rays(1 << 20, seed=6)  # the same workload at a size that fills the GPU
    table, last = {}, {}
    steps = args.steps
    for alg in PT_ALGS:
        rtb200.perf_test(xy, wl["radius"], wl["angle"], wl["arch_seg"], wl["path_seg"], alg)  # warm-up (context, first launch)
        runs = [rtb200.perf_test(xy, wl["radius"], wl["angle"], wl["arch_seg"], wl["path_seg"], alg) for _ in range(steps)]
        last.update({f"{alg}_{k}": runs[-1][k] for k in ("reached", "depth", "last_id", "last_pos")})
        b = rtb200.perf_test(big, wl["radius"], wl["angle"], wl["arch_seg"], wl["path_seg"], alg)
        table[alg] = {"trace_ms": float(np.mean([r["trace_ms"] for r in runs])), "build_ms": runs[-1]["build_ms"],
                      "preprocess_ms": runs[-1]["preprocess_ms"], "total_rays": int(runs[-1]["total_rays"]),
                      "published_trace_ms": PT_PUBLISHED_TRACE_MS[alg],
                      "at_1M_rays": {"trace_ms": b["trace_ms"], "Mrays/s": b["total_rays"] / b["trace_ms"] / 1e3, "total_rays": int(b["total_rays"])}}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    cpu = None
    if not args.no_cpu:
        try:
            from oracle import oracle_py as O
            which = "ref_pt" if O.available("ref_pt") else "oracle"
            r = O.bounce(which, xy, wl["radius"], wl["angle"], wl["arch_seg"], wl["path_seg"], "sah", 200, threads=1, pt_builders=True)
            g = rtb200.perf_test(xy, wl["radius"], wl["angle"], wl["arch_seg"], wl["path_seg"], "sah")
            same = bool(np.array_equal(r["reached"], g["reached"]) and np.array_equal(r["depth"], g["depth"]) and np.array_equal(r["last_id"], g["last_id"]))
            cpu = {"value": r["trace_ms"], "unit": "ms", "cores": 1, "kind": "reference" if which == "ref_pt" else "port",
                   "sample": "the same 1000 rays, k-d SAH, single thread as the reference program runs it", "prepare_ms": r["prepare_ms"],
                   "parity_checked": same}
            if not same:
                raise SystemExit("PerformanceTest parity check failed: per-ray results differ from the reference program")
        except SystemExit:
            raise
        except Exception as e:
            cpu = {"error": str(e)}
    v = table["sah"]["trace_ms"]
    emit({"metric": "PerformanceTest trace ms (k-d SAH; 1000 random rays, <= 200 mirror bounces)", "value": v, "unit": "ms", "n_gpus": 1,
          "steps": steps, "warmup": 1, "ms_per_step": v, "higher_is_better": False, "scaling": "strong",
          "vs_baseline": v / PT_PUBLISHED_TRACE_MS["sah"], "dtype": "f32", "data": "synthetic",
          "config": {"workload": wl_name, "description": wl["desc"], "table": table,
                     "note": "trace_ms is the kernel's CUDA-event time as rt::PerformanceTest reports it; 1000 rays occupy 8 CTAs of one GPU, so the "
                             "number is the latency of the longest bounce chain -- at_1M_rays is the same loop at a size that fills the device"},
          "roofline": None, "cpu_baseline": cpu,
          "e2e": {"value": v, "unit": "ms", "h2d_bytes_per_step": int(xy.nbytes), "d2h_bytes_per_step": int(wl["rays"] * 24)},
          "gpu_launches": steps * len(PT_ALGS)})


# ---- the B200 arm ----------------------------------------------------------------------------------
def moved_camera(cam, k):
    import rtb200
    c = rtb200.Camera.from_buffer_copy(cam)
    c.eye[2] = cam.eye[2] - 0.25 * (k + 1)  # dolly into the tunnel, a quarter unit per frame
    return c


def run_b200(args, wl_name):
    import torch
    import rtb200

    wl = WORKLOADS[wl_name]
    if wl.get("kind") == "pt":
        return run_pt(args, wl_name)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        host_group = dist.new_group(backend="gloo")  # waits on the HOST: an idle rank parked in an NCCL barrier keeps a kernel
        #                                              spinning on its GPU, which time-slices against rank 0's context there
    dev_t = torch.device("cuda", local)

    def host_barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier(group=host_group)

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev_t)
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev_t)
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    W, H, spp = wl["width"], wl["height"], wl["samples"]
    mc = wl["preset"] <= 3 and wl.get("setting") != "simple"
    t0 = time.perf_counter()
    scene = rtb200.PresetScene(wl["preset"], wl["algorithm"], wl["segments"])
    host_build_s = time.perf_counter() - t0
    setting = rtb200.make_setting(wl["setting"]) if "setting" in wl else scene.setting
    ctx = rtb200.Context(local)
    dscene = ctx.upload(scene.flat)
    col_block = COL_BLOCK if (world >= max(COL_MIN_WORLD, 2) and COL_BLOCK > 0 and W % (world * COL_BLOCK) == 0) else 0
    # Monte-Carlo frames whose pixel shards would not fill a GPU for more than a few waves of warps shard over SAMPLES instead:
    # every rank renders every pixel with spp / N of the samples (RNG keyed by pixel and sample index) and one NCCL reduce (sum)
    # onto rank 0 assembles the frame (SURVEY 8e).  One wave = 148 SMs x 32 resident warps = 4,736 tiles.
    sample_sharded = (mc and world > 1 and spp >= world and args.mc_shard != "pixels"
                      and (args.mc_shard == "samples" or (W * H // 32) // world < 8 * 4736))
    if sample_sharded:
        col_block = 0
    peer = world > 1 and args.gather in ("peer", "scatter") and not sample_sharded
    scatter = peer and args.gather == "scatter"  # render into a local shard, then ONE streaming copy into the owner's frame
    layout = rtb200.LAYOUT_GLOBAL if (peer and not scatter) else rtb200.LAYOUT_ROWMAJOR
    if sample_sharded:
        s_first, s_count = rtb200.sample_shard(spp, rank, world)
        frame = rtb200.make_frame(W, H, samples=spp, seed=0, sample_first=s_first, sample_count=s_count)
        shard = frame
    else:
        frame = rtb200.make_frame(W, H, samples=spp, seed=0, rank=rank, world=world, row_block=ROW_BLOCK, col_block=col_block, layout=layout)
        shard = rtb200.make_frame(W, H, samples=spp, seed=0, rank=rank, world=world, row_block=ROW_BLOCK, col_block=col_block)
    Wl = rtb200.shard_width(shard)  # width of this rank's local image
    rows = rtb200.shard_rows(shard)
    rows_max = int(allmax(rows))
    # a dedicated (non-default) torch stream: the kernels, the NCCL calls and the timing events all live on it
    tstream = torch.cuda.Stream(device=dev_t)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream

    frame_bytes = W * H * 3 * 4
    owner_frame = None   # rank 0's device frame (rtb_device_alloc), mapped into the peers through CUDA IPC
    mapped = None
    if world == 1 or sample_sharded:
        image = torch.zeros((H, W, 3), dtype=torch.float32, device=dev_t)
        target = image.data_ptr()
    elif peer:
        handle = [None]
        if rank == 0:
            owner_frame = ctx.device_alloc(frame_bytes)
            handle[0] = ctx.ipc_export(owner_frame)
        dist.broadcast_object_list(handle, src=0)
        mapped = owner_frame if rank == 0 else ctx.ipc_open(handle[0])
        target = mapped
        if scatter:
            local_buf = torch.zeros((rows_max, Wl, 3), dtype=torch.float32, device=dev_t)
            target = local_buf.data_ptr()
        token = torch.zeros(1, dtype=torch.int32, device=dev_t)
    else:
        image = torch.zeros((H, W, 3), dtype=torch.float32, device=dev_t)
        local_buf = torch.zeros((rows_max, Wl, 3), dtype=torch.float32, device=dev_t)
        gathered = torch.zeros((world, rows_max, Wl, 3), dtype=torch.float32, device=dev_t)
        target = local_buf.data_ptr()

    def unshard():
        if col_block:
            rtb200.unshard_cols_device(ctx, gathered.data_ptr(), image.data_ptr(), W, H, world, ROW_BLOCK, col_block, stream)
        else:
            rtb200.unshard_device(ctx, gathered.data_ptr(), image.data_ptr(), W, H, world, ROW_BLOCK, rows_max, stream)
    flush = torch.empty(384 * 1024 * 1024, dtype=torch.uint8, device=dev_t)  # > 126 MB L2

    def render(cam=None, want_stats=False, fr=None):
        return dscene.render_device(cam or scene.camera, setting, fr or frame, target, stream, want_stats=want_stats)

    def close_step():
        if world == 1:
            return
        if sample_sharded:
            dist.reduce(image, dst=0, op=dist.ReduceOp.SUM)  # rank 0: the frame; every sample carries the weight 1 / spp
        elif peer:
            if scatter:
                ctx.scatter_shard_device(local_buf.data_ptr(), mapped, shard, stream)
            dist.all_reduce(token)  # every rank's tiles are in the owner's frame when this completes
        else:
            dist.all_gather_into_tensor(gathered.view(world * rows_max, Wl, 3), local_buf)
            unshard()

    def step():
        render()
        close_step()

    # ray / test / step counts of one frame (deterministic), outside the timed region
    cframe = rtb200.Frame.from_buffer_copy(frame)
    cframe.counters = 1
    cst = render(want_stats=True, fr=cframe)
    rays_frame = allsum(cst["n_rays"])
    tests_frame = allsum(cst["n_tri_tests"])
    steps_frame = allsum(cst["n_steps"])

    # ---- first frame of a view (fresh schedule: raster order, one throughput kernel) and a moving camera (order kept,
    # latency tiers off), device-resident, this rank's kernels; L2 flushed before each
    first_ms, moving_ms = [], []
    for _ in range(3):
        ctx.forget_schedule()
        flush.zero_()
        first_ms.append(render(want_stats=True)["kernel_ms"])
    if not mc:
        render(); render()
        for k in range(4):
            flush.zero_()
            moving_ms.append(render(cam=moved_camera(scene.camera, k), want_stats=True)["kernel_ms"])
    first_frame_ms = allmax(float(np.median(first_ms)))
    moving_camera_ms = allmax(float(np.mean(moving_ms))) if moving_ms else None

    ctx.forget_schedule()
    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    barrier()

    # kernels of this library per step, as counted by the library for this frame (rtb_stats.n_launches): the render
    # kernels (1-3: throughput walk + up to two latency tiers) + 3 tile-order kernels (+ the unshard kernel with --gather nccl)
    kst = render(want_stats=True)
    launches_per_step = int(kst["n_launches"]) + (1 if (world > 1 and (not peer or scatter)) else 0)
    close_step()

    sampler = ClockSampler(local) if rank == 0 else None
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    if sampler:
        sampler.start()
    for i in range(args.steps):
        flush.zero_()  # L2 flush between timed iterations (not timed)
        ev[i][0].record()
        kev[i][0].record()
        render()
        kev[i][1].record()
        close_step()
        ev[i][1].record()
    barrier()
    clocks = sampler.stop() if sampler else None
    total_ms = allmax(sum(a.elapsed_time(b) for a, b in ev))
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    kernel_ms_max = allmax(kernel_ms)
    ms_per_step = total_ms / args.steps
    value = rays_frame / ms_per_step / 1e3  # Mrays/s, whole job

    # ---- what was rendered is checked, outside the timed region ----
    verified = None
    gpu_image = None
    if world == 1:
        torch.cuda.synchronize()
        gpu_image = image.cpu().numpy()
    elif sample_sharded:
        barrier()
        step()  # one more frame so that rank 0's buffer holds exactly one reduced frame (the timed loop reduced in place over it too)
        torch.cuda.synchronize()
        if rank == 0:  # float sums of the same samples in another order: equal within rounding, not bit for bit
            assembled = image.cpu().numpy()
            alone, _ = dscene.render(scene.camera, setting, rtb200.make_frame(W, H, samples=spp, seed=0))
            verified = bool(np.allclose(assembled, alone, rtol=2e-5, atol=1e-6))
            if not verified:
                raise SystemExit("sample-sharded frame differs from the single-GPU frame beyond float rounding")
            gpu_image = assembled
        barrier()
    elif peer:
        barrier()
        if rank == 0:  # the assembled frame in the owner's memory == the frame one GPU renders alone, bit for bit
            assembled = ctx.device_download(owner_frame, np.zeros((H, W, 3), np.float32))
            alone, _ = dscene.render(scene.camera, setting, rtb200.make_frame(W, H, samples=spp, seed=0))
            verified = bool(np.array_equal(assembled.view(np.uint32), alone.view(np.uint32)))
            if not verified:
                raise SystemExit("assembled multi-GPU frame differs from the single-GPU frame")
            gpu_image = assembled
        barrier()
    if args.dump_outputs and rank == 0:  # the frame of the last timed step (--gather nccl: the unsharded frame on rank 0)
        dump_outputs(args.dump_outputs, {}, gpu_image if gpu_image is not None else image.cpu().numpy())

    # ---- e2e: host buffers through the C ABI; scene H2D + render + the ASSEMBLED frame in one page-locked host buffer, per step
    e2e_steps = max(3, min(args.steps, 10))
    e2e = None
    if world == 1:
        pinned = rtb200.PinnedArray((H, W, 3))  # rtb_host_alloc: page-locked host framebuffer
        h2d = dscene.upload_bytes

        def e2e_step(out=pinned.array, fr=rtb200.make_frame(W, H, samples=spp, seed=0)):
            d = ctx.upload(scene.flat)
            d.render(scene.camera, setting, fr, out=out)
            d.close()

        def timed_e2e(*a):
            e2e_step(*a)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            for _ in range(e2e_steps):
                e2e_step(*a)
            torch.cuda.synchronize()
            return (time.perf_counter() - t1) * 1e3 / e2e_steps

        e2e_pageable_ms = timed_e2e()  # the flat scene's arrays in pageable memory: the upload stages them (one host pass over the scene)
        scene.pin()                    # ... page-locked where they lie (rtb_host_register): the upload copies H2D straight out of them
        e2e_ms = timed_e2e()
        # the same call with the reference's 8-bit output stage on the GPU (3 bytes per pixel come back)
        pinned8 = rtb200.PinnedArray(((H * W * 3 + 3) // 4,))
        host8 = pinned8.array.view(np.uint8)[: H * W * 3].reshape(H, W, 3)
        f8 = rtb200.make_frame(W, H, samples=spp, seed=0, layout=rtb200.OUTPUT_RGB8)
        e2e8_ms = timed_e2e(host8, f8)
        scene.unpin()
        e2e = {"value": rays_frame / e2e_ms / 1e3, "unit": "Mrays/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(frame_bytes),
               "ms_per_step": e2e_ms, "steps": e2e_steps,
               "path": "rtb_scene_upload (H2D out of the caller's page-locked scene arrays, rtb_flat_scene.arrays_page_locked) + rtb_render (the kernels store the float "
                       "frame straight into the caller's page-locked host buffer over PCIe) + rtb_scene_free, per step",
               "pageable_scene_arrays": {"value": rays_frame / e2e_pageable_ms / 1e3, "ms_per_step": e2e_pageable_ms,
                                         "note": "same step with the scene arrays in pageable memory (the upload stages them in its page-locked ring first)"},
               "rgb8_output_stage": {"value": rays_frame / e2e8_ms / 1e3, "ms_per_step": e2e8_ms, "d2h_bytes_per_step": int(H * W * 3),
                                     "note": "same call with RTB_OUTPUT_RGB8: saturate + (int)(c*255) on the GPU as the reference's Render ends (MainWindow.cpp:305-311)"}}
    else:
        host_barrier()
        if rank == 0:  # ONE host thread drives all N devices (rtb_multi_*); the other ranks' processes are idle meanwhile (parked on the host)
            multi = rtb200.MultiContext(world)
            pinned = rtb200.PinnedArray((H, W, 3))
            scene.pin()  # scene arrays page-locked where they lie: every device copies H2D straight out of them
            mframe = rtb200.make_frame(W, H, samples=spp, seed=0, row_block=ROW_BLOCK)

            phases = []

            def e2e_step():
                ta = time.perf_counter()
                d = multi.upload(scene.flat)
                tb = time.perf_counter()
                _, mst = d.render(scene.camera, setting, mframe, out=pinned.array)
                tc = time.perf_counter()
                h = d.upload_bytes
                d.close()
                phases.append(((tb - ta) * 1e3, (tc - tb) * 1e3, mst["kernel_ms"]))
                return h

            for _ in range(3):
                h2d = e2e_step()
            del phases[:]
            t1 = time.perf_counter()
            for _ in range(e2e_steps):
                e2e_step()
            e2e_ms = (time.perf_counter() - t1) * 1e3 / e2e_steps
            ph = np.asarray(phases).mean(axis=0)
            same = bool(gpu_image is not None and (np.allclose(pinned.array, gpu_image, rtol=2e-5, atol=1e-6) if sample_sharded
                                                   else np.array_equal(pinned.array.view(np.uint32), gpu_image.view(np.uint32))))
            e2e = {"value": rays_frame / e2e_ms / 1e3, "unit": "Mrays/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(frame_bytes),
                   "ms_per_step": e2e_ms, "steps": e2e_steps, "assembled_host_frame_verified": same if gpu_image is not None else None,
                   "phases_ms": {"upload_all_devices": float(ph[0]), "render_all_devices": float(ph[1]), "slowest_device_kernels": float(ph[2])},
                   "path": f"rank 0's host thread drives all {world} devices: rtb_multi_scene_upload (H2D to every device, side by side, out of the page-locked scene arrays) + rtb_multi_render (every device stores "
                           "its tiles straight into ONE page-locked host frame over its own PCIe link) + rtb_multi_scene_free, per step"}
            multi.close()
            scene.unpin()
        host_barrier()

    # ---- roofline of the frame's kernels: warp-instruction issue
    peaks, peak_kind = measured_peaks()
    counts, counts_source = issue_counts(wl_name)
    clock_mhz = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)
    peak_ginst = N_SM * SCHEDULERS * clock_mhz * 1e-3  # G warp-instructions / s
    roofline = {"bound": "issue", "unit": "Gwarp-inst/s", "peak": peak_ginst, "achieved": None, "frac": None, "traffic": None,
                "peak_source": f"{N_SM} SMs x {SCHEDULERS} schedulers x the median SM clock sampled during the timed region ({clock_mhz:.0f} MHz)",
                "kernel_ms": kernel_ms}
    if counts and world == 1:
        winst = counts["warp_inst"]
        roofline.update({"achieved": winst / (kernel_ms * 1e-3) / 1e9, "frac": winst / (kernel_ms * 1e-3) / 1e9 / peak_ginst,
                         "warp_inst_per_frame": winst, "kernels": counts.get("kernels"),
                         "thread_inst_per_warp_inst": counts.get("thread_inst_per_warp_inst"),
                         "useful_lane_frac": (winst / (kernel_ms * 1e-3) / 1e9 / peak_ginst) * counts.get("thread_inst_per_warp_inst", 32.0) / 32.0
                         if counts.get("thread_inst_per_warp_inst") else None,
                         "ncu": {k: counts.get(k) for k in ("issue_active_pct", "ipc_per_sm", "l1_hit_pct", "duration_ms_under_ncu")},
                         "traffic": counts.get("dram_bytes"), "compulsory_bytes": int(frame_bytes) if not mc else int(frame_bytes),
                         "counts_source": counts_source})
    elif world > 1:
        # a rank's shard: the instruction counts of rank 0's 1/N shard (ncu capture of the same frame rendered as a shard on one GPU),
        # against the slowest rank's kernel time -- all ranks hold the same mix of tiles (column-block shards)
        shard, shard_source = issue_counts(f"{wl_name}_shard_1of{world}")
        if shard:
            winst = shard["warp_inst"]
            roofline.update({"achieved": winst / (kernel_ms * 1e-3) / 1e9, "frac": winst / (kernel_ms * 1e-3) / 1e9 / peak_ginst,
                             "warp_inst_per_shard": winst, "thread_inst_per_warp_inst": shard.get("thread_inst_per_warp_inst"),
                             "per": "rank (one GPU's issue peak against one shard's instructions and the slowest rank's kernel time)",
                             "traffic": shard.get("dram_bytes"), "compulsory_bytes": int(frame_bytes // world), "counts_source": shard_source})
    # HBM side of the same kernels, for the record: algorithmic bytes (DESIGN.md section 5: 8 B per visited cell / k-d node, 4 B index + 36 B
    # vertices per triangle test, 12 B normal + 4 B material per ray, 12 B framebuffer per pixel) are served by L1 / L2; DRAM sees `traffic`
    algo_bytes = 8 * cst["n_steps"] + 40 * cst["n_tri_tests"] + 16 * cst["n_rays"] + 12 * rows * Wl
    roofline["hbm"] = {"algorithmic_bytes_per_launch": algo_bytes, "bytes_per_ray": algo_bytes / max(cst["n_rays"], 1),
                       "algorithmic_GBs": algo_bytes / (kernel_ms * 1e-3) / 1e9, "peak_GBs": peaks["hbm_gbs"], "peak_source": peak_kind,
                       "dram_GBs": (roofline["traffic"] / (kernel_ms * 1e-3) / 1e9) if roofline["traffic"] else None,
                       "dram_frac_of_peak": (roofline["traffic"] / (kernel_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]) if roofline["traffic"] else None}

    # ---- other preset configs, one device-resident frame each, not part of `value`
    others = {}
    if not args.no_extras and world == 1:
        for name in EXTRAS:
            if name == wl_name:
                continue
            o = WORKLOADS[name]
            try:
                s2 = rtb200.PresetScene(o["preset"], o["algorithm"], o["segments"])
                set2 = rtb200.make_setting(o["setting"]) if "setting" in o else s2.setting
                d2 = ctx.upload(s2.flat)
                buf = torch.empty((o["height"], o["width"], 3), dtype=torch.float32, device=dev_t)
                f2 = rtb200.make_frame(o["width"], o["height"], samples=o["samples"])
                ctx.forget_schedule()
                first = d2.render_device(s2.camera, set2, f2, buf.data_ptr(), stream, want_stats=True)
                best = None
                for _ in range(5):
                    st = d2.render_device(s2.camera, set2, f2, buf.data_ptr(), stream, want_stats=True)
                    best = st if best is None or st["kernel_ms"] < best["kernel_ms"] else best
                others[name] = {"Mrays/s": best["n_rays"] / best["kernel_ms"] / 1e3, "ms": best["kernel_ms"], "first_frame_ms": first["kernel_ms"],
                                "rays": best["n_rays"], "host_build_s": s2.build_ms / 1e3}
                d2.close(); s2.close(); del buf
            except Exception as e:  # report, do not hide
                others[name] = {"error": str(e)}

    # ---- the reference's Render() on the host cores, same frame; and the parity of what the GPU rendered
    cpu, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            fit, est = cpu_repeats(wl)
            res = cpu_reference(wl, repeat=fit, warmup=0, image=True)
            ms = float(res["ms"].mean())
            cpu = {"value": res["rays"] / ms / 1e3, "unit": "Mrays/s", "cores": res["cores"], "kind": res["kind"],
                   "sample": f"the whole {W}x{H} frame at {spp} spp, mean of {fit} Render() call(s)", "render_s": ms / 1e3, "prepare_s": res["prepare_ms"] / 1e3}
            ref = res["image"]
            if ref is not None and gpu_image is not None:
                if mc:  # different random streams (erand48 per row vs Philox per pixel): image-mean luminance only; the tests hold the full criteria
                    rel = abs(float(gpu_image.mean()) - float(ref.mean())) / float(ref.mean())
                    parity = {"checked": "statistical", "image_mean_rel_diff": rel, "ok": bool(rel < 0.01)}
                else:
                    err = np.abs(gpu_image - ref)
                    ok = bool((err <= 1e-5 * np.abs(ref) + 1e-7).all() and rays_frame == res["rays"])
                    exact = float((gpu_image.view(np.uint32) == ref.view(np.uint32)).mean())
                    parity = {"checked": "every pixel of the timed frame vs the CPU checker at 1e-5 relative; ray counts equal", "ok": ok,
                              "bit_exact_fraction": exact, "max_abs_err": float(err.max()), "rays_gpu": rays_frame, "rays_cpu": res["rays"]}
                if not parity["ok"]:
                    raise SystemExit(f"parity check failed: {parity}")
        except SystemExit:
            raise
        except Exception as e:
            cpu = {"error": str(e)}

    launches_total = allsum(launches_per_step * args.steps)
    if rank == 0:
        sharding = (f"column blocks of {col_block} pixels, rotated every {ROW_BLOCK} rows, dealt round-robin to {world} rank(s)" if col_block
                    else f"tile rows, blocks of {ROW_BLOCK} rows dealt round-robin to {world} rank(s)")
        if world > 1:
            if sample_sharded:
                sharding = f"SAMPLE shards: every rank renders every pixel with {spp} / {world} of the samples; NCCL reduce (sum) onto rank 0 every step"
            else:
                sharding += ("; every rank stores its tiles straight into rank 0's device frame over NVLink (CUDA IPC mapping, RTB_LAYOUT_GLOBAL), "
                             "a one-word NCCL all-reduce closes the step" if (peer and not scatter) else
                             "; every rank renders into a local shard and moves it with one streaming copy kernel into rank 0's device frame over NVLink (CUDA IPC mapping), "
                             "a one-word NCCL all-reduce closes the step" if scatter else "; NCCL all_gather_into_tensor + unshard kernel every step")
        line = {"metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": wl_name, "description": wl["desc"], "rays_per_step": rays_frame,
                           "tri_tests_per_step": tests_frame, "traversal_steps_per_step": steps_frame, "sharding": sharding,
                           "timing": "steady state of one view (tile order + latency tiers learnt from the previous frames of the same view); "
                                     "first_frame_ms / moving_camera_ms are the same frame without that state",
                           "l2": "flushed between timed iterations (384 MiB memset, untimed)",
                           "host_build_s": host_build_s, "scene_device_bytes": dscene.device_bytes, "scene_upload_bytes": dscene.upload_bytes},
                "first_frame_ms": first_frame_ms, "moving_camera_ms": moving_camera_ms,
                "roofline": roofline, "cpu_baseline": cpu, "parity_checked": bool(parity and parity["ok"]), "parity": parity,
                "assembled_frame_verified": verified, "e2e": e2e,
                "gpu_launches": int(launches_total),
                "kernel_ms_max_over_ranks": kernel_ms_max, "clocks": clocks, "others": others}
        emit(line)
    if mapped is not None and rank != 0:
        ctx.ipc_close(mapped)
    if dist:
        dist.barrier()
    if owner_frame is not None:
        ctx.device_free(owner_frame)
    dscene.close(); scene.close(); ctx.close()
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="p5_sah_4k", choices=sorted(WORKLOADS))
    ap.add_argument("--gather", default="peer", choices=["peer", "scatter", "nccl"])
    ap.add_argument("--mc-shard", default="auto", choices=["auto", "samples", "pixels"])
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 arm (--impl b200)")
    sys.dont_write_bytecode = True  # the run leaves the tree as it found it (it may be read-only)
    # stdout carries exactly one JSON line: file descriptor 1 is pointed at stderr for the duration of the run
    # (NCCL prints its version banner to stdout whatever NCCL_DEBUG_FILE says) and emit() writes to the saved one
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, args.workload)
    else:
        run_b200(args, args.workload)


if __name__ == "__main__":
    main()
