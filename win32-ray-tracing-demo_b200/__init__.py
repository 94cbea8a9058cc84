"""rtb200 -- Python harness over the C ABI (include/rtb.h) and the C++ host API (host/rt.h).

The product is the two in-tree shared libraries; this module only binds them with ctypes for the
tests, bench.py and torch.distributed plumbing.  The directory name is not a Python identifier, so
import it through `rtb200.py` at the repo root (`import rtb200`).

There is no CPU fallback anywhere below: every compute call goes to librtb200.so's CUDA kernels
and raises RtbError when the library or a CUDA device is missing.
"""
import ctypes as C
import os

import numpy as np

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CUDA_LIB = os.path.join(PKG, os.environ.get("RTB_CUDA_LIB_NAME", "librtb200.so"))  # RTB_CUDA_LIB_NAME: an experiment build (tools/)
HOST_LIB = os.path.join(PKG, "librtb200_host.so")

ALGORITHMS = {"linear": 0, "rgrid": 1, "fgrid": 2, "kd": 3, "sah": 4, "convex": 5, "convexsimple": 6}
STAT_NAMES = ["n_top", "n_tris", "grid_x", "grid_y", "grid_z", "cells_nonempty", "cell_entries",
              "cell_max", "kd_nodes", "kd_leaves", "kd_leaf_refs", "kd_max_depth"]
LAYOUT_ROWMAJOR, LAYOUT_REFERENCE, LAYOUT_GLOBAL, OUTPUT_RGB8, OUTPUT_MOMENTS = 0, 1, 2, 4, 8
IPC_HANDLE_BYTES = 64
PRIM_PLANE, PRIM_SPHERE, PRIM_TRIANGLES, PRIM_TUNNEL, PRIM_MESH = 0, 1, 2, 3, 4  # rtb_prim.type
MESH_REBUILD, MESH_REFIT = 0, 1  # rtb_scene_mesh_update flags
CUDA_STREAM_LEGACY = 1  # cudaStreamLegacy
QUERY_CLOSEST, QUERY_ANY = 0, 1  # rtb_query_rays / rtb_query_points flags
QUERY_PAIRS = 2  # rtb_query_triangles: every intersecting pair (QUERY_ANY: a flag per triangle)


class RtbError(RuntimeError):
    pass


# ---- ctypes mirrors of include/rtb.h ---------------------------------------------------------
class Material(C.Structure):
    _fields_ = [("kind", C.c_int32), ("diffusiveness", C.c_float), ("reflectiveness", C.c_float),
                ("refractiveness", C.c_float), ("refractive_index", C.c_float), ("a", C.c_float * 3),
                ("b", C.c_float * 3), ("scale", C.c_float), ("p", C.c_float), ("dir", C.c_int32),
                ("pad_", C.c_int32 * 2)]


class Prim(C.Structure):
    _fields_ = [("type", C.c_int32), ("material", C.c_int32), ("base_id", C.c_int32),
                ("first", C.c_int32), ("count", C.c_int32), ("v", C.c_float * 7)]


class KdNode(C.Structure):
    _fields_ = [("a", C.c_uint32), ("b", C.c_uint32)]


class BvhNode(C.Structure):
    """rtb_bvhnode: boxes lo/hi [child][axis] of the two children, child links (>= 0 inner node, < 0 leaf position ~c)."""
    _fields_ = [("lo", (C.c_float * 3) * 2), ("hi", (C.c_float * 3) * 2), ("child", C.c_int32 * 2), ("pad_", C.c_int32 * 2)]


class CellWord(C.Structure):
    _fields_ = [("bits", C.c_uint32), ("rank", C.c_uint32)]


class FlatScene(C.Structure):
    _fields_ = [
        ("n_prims", C.c_int32), ("prims", C.POINTER(Prim)),
        ("n_materials", C.c_int32), ("materials", C.POINTER(Material)),
        ("n_top", C.c_int32),
        ("n_loose", C.c_int32), ("loose_tri", C.POINTER(C.c_float)),
        ("n_tris", C.c_int32), ("tri", C.POINTER(C.c_float)), ("tri_material", C.POINTER(C.c_int32)),
        ("accel", C.c_int32),
        ("grid_origin", C.c_float * 3), ("grid_cell", C.c_float * 3), ("grid_dims", C.c_int32 * 3),
        ("grid_build_resolution", C.c_int32),
        ("n_cellwords", C.c_int64), ("grid_words", C.POINTER(CellWord)),
        ("n_cells_used", C.c_int64), ("grid_cell_start", C.POINTER(C.c_uint32)),
        ("n_cell_refs", C.c_int64), ("grid_cell_tris", C.POINTER(C.c_uint32)),
        ("kd_min", C.c_float * 3), ("kd_max", C.c_float * 3),
        ("n_kd_nodes", C.c_int32), ("kd_nodes", C.POINTER(KdNode)),
        ("n_kd_refs", C.c_int64), ("kd_leaf_tris", C.POINTER(C.c_uint32)),
        ("n_cx_path", C.c_int32), ("cx_frames", C.POINTER(C.c_float)),
        ("n_cx_edges", C.c_int32), ("cx_edges", C.POINTER(C.c_float)),
        ("cx_width", C.c_float), ("cx_height", C.c_float),
        ("cx_table_size", C.c_int32), ("cx_round_bins", C.c_int32),
        ("cx_cell_status", C.POINTER(C.c_uint8)), ("cx_cell_range", C.POINTER(C.c_int16)),
        ("cx_order", C.POINTER(C.c_uint16)),
        ("grid_build_exact", C.c_int32),
        ("kd_build_leaf_size", C.c_int32), ("kd_build_max_depth", C.c_int32), ("kd_build_candidates", C.c_int32),
        ("arrays_page_locked", C.c_int32),
    ]

    def arrays(self):
        """(address, bytes) of every array rtb_scene_upload copies for this scene (include/rtb.h: rtb_flat_scene)."""
        def a(ptr, n, elem):
            return (C.cast(ptr, C.c_void_p).value, int(n) * elem) if ptr and n > 0 else None
        out = [a(self.loose_tri, self.n_loose, 48), a(self.tri, self.n_tris, 48), a(self.tri_material, self.n_tris, 4)]
        if self.accel in (ALGORITHMS["rgrid"], ALGORITHMS["fgrid"]) and self.grid_words:
            out += [a(self.grid_words, self.n_cellwords, 8), a(self.grid_cell_start, self.n_cells_used + 1, 4),
                    a(self.grid_cell_tris, self.n_cell_refs, 4)]
        if self.accel in (ALGORITHMS["kd"], ALGORITHMS["sah"]) and self.kd_nodes:
            out += [a(self.kd_nodes, self.n_kd_nodes, 8), a(self.kd_leaf_tris, self.n_kd_refs, 4)]
        return [x for x in out if x]


class Camera(C.Structure):
    _fields_ = [("eye", C.c_float * 3), ("front", C.c_float * 3), ("up", C.c_float * 3),
                ("right", C.c_float * 3), ("xcenter", C.c_float), ("fov_scale", C.c_float),
                ("forward", C.c_float)]


class RenderSetting(C.Structure):
    _fields_ = [("enable_monte_carlo", C.c_int32), ("max_depth", C.c_int32),
                ("termination_depth", C.c_int32), ("single_tracing_depth", C.c_int32)]


INT_MAX = 2 ** 31 - 1
SETTINGS = {  # reference RenderSetting.h:40-78
    "simple": (0, 20, INT_MAX, 0), "default": (1, INT_MAX, 5, 2),
    "highspeed": (1, 6, 2, 0), "highquality": (1, 8, INT_MAX, INT_MAX),
}


class Frame(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("samples", C.c_int32),
                ("seed", C.c_uint64), ("rank", C.c_int32), ("world", C.c_int32),
                ("row_block", C.c_int32), ("layout", C.c_int32), ("counters", C.c_int32),
                ("col_block", C.c_int32), ("sample_first", C.c_int32), ("sample_count", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("n_rays", C.c_int64), ("n_tri_tests", C.c_int64), ("n_steps", C.c_int64),
                ("n_local_rows", C.c_int64), ("kernel_ms", C.c_float), ("total_ms", C.c_float),
                ("n_launches", C.c_int32), ("pad_", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "pad_"}


ABI_SYMBOLS = ["rtb_init", "rtb_shutdown", "rtb_last_error", "rtb_abi_version", "rtb_shard_rows", "rtb_shard_width",
               "rtb_unshard_cols_device",
               "rtb_host_alloc", "rtb_host_free", "rtb_host_register", "rtb_host_unregister",
               "rtb_scene_upload", "rtb_scene_free", "rtb_scene_device_bytes", "rtb_scene_upload_bytes", "rtb_scene_grid_hash", "rtb_scene_kd_download", "rtb_scene_mesh_download", "rtb_scene_mesh_update", "rtb_render",
               "rtb_render_device", "rtb_unshard_device", "rtb_trace_primary", "rtb_intersect_rays", "rtb_bounce_rays",
               "rtb_selftest_pretest", "rtb_kd_validate", "rtb_forget_schedule", "rtb_set_progress", "rtb_multi_set_progress",
               "rtb_device_alloc", "rtb_device_free", "rtb_device_download", "rtb_ipc_export", "rtb_ipc_open", "rtb_ipc_close", "rtb_scatter_shard_device",
               "rtb_multi_init", "rtb_multi_shutdown", "rtb_multi_count", "rtb_multi_ctx", "rtb_multi_last_error",
               "rtb_multi_scene_upload", "rtb_multi_scene_free", "rtb_multi_scene_upload_bytes", "rtb_multi_render",
               "rtb_multi_scene_mesh_update", "rtb_query_rays", "rtb_query_points",
               "rtb_scene_mesh_moments", "rtb_query_winding", "rtb_query_triangles"]

_cuda = None
_host = None


def cuda_lib():
    """librtb200.so; raises RtbError (never falls back) when it has not been built."""
    global _cuda
    if _cuda is None:
        if not os.path.exists(CUDA_LIB):
            raise RtbError(f"{CUDA_LIB} is missing: run `python __graft_entry__.py build` (there is no CPU fallback)")
        lib = C.CDLL(CUDA_LIB, mode=C.RTLD_GLOBAL)
        vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
        lib.rtb_init.argtypes = [C.c_int, C.POINTER(vp)]
        lib.rtb_shutdown.argtypes = [vp]
        lib.rtb_last_error.argtypes = [vp]
        lib.rtb_last_error.restype = C.c_char_p
        lib.rtb_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
        lib.rtb_host_free.argtypes = [vp]
        lib.rtb_host_register.argtypes = [vp, C.c_size_t]
        lib.rtb_host_unregister.argtypes = [vp]
        lib.rtb_shard_rows.argtypes = [C.POINTER(Frame)]
        lib.rtb_shard_rows.restype = i64
        lib.rtb_shard_width.argtypes = [C.POINTER(Frame)]
        lib.rtb_shard_width.restype = i64
        lib.rtb_scene_upload.argtypes = [vp, C.POINTER(FlatScene), C.POINTER(vp)]
        lib.rtb_scene_free.argtypes = [vp, vp]
        lib.rtb_scene_device_bytes.argtypes = [vp]
        lib.rtb_scene_device_bytes.restype = i64
        lib.rtb_scene_upload_bytes.argtypes = [vp]
        lib.rtb_scene_upload_bytes.restype = i64
        lib.rtb_scene_grid_hash.argtypes = [vp, vp, C.POINTER(C.c_uint64), C.POINTER(C.c_int64)]
        lib.rtb_scene_grid_hash.restype = C.c_int
        lib.rtb_scene_kd_download.argtypes = [vp, vp, vp, i64, vp, i64, C.POINTER(C.c_int64), C.POINTER(C.c_float)]
        lib.rtb_scene_mesh_download.argtypes = [vp, vp, i32, vp, i64, vp, i64, C.POINTER(C.c_int64)]
        lib.rtb_scene_mesh_update.argtypes = [vp, vp, i32, vp, i64, i32, vp]
        lib.rtb_render.argtypes = [vp, vp, C.POINTER(Camera), C.POINTER(RenderSetting), C.POINTER(Frame), vp,
                                   C.POINTER(Stats)]
        lib.rtb_render_device.argtypes = [vp, vp, C.POINTER(Camera), C.POINTER(RenderSetting), C.POINTER(Frame),
                                          vp, vp, C.POINTER(Stats)]
        lib.rtb_unshard_device.argtypes = [vp, vp, vp, i32, i32, i32, i32, i64, vp]
        lib.rtb_unshard_cols_device.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, vp]
        lib.rtb_trace_primary.argtypes = [vp, vp, C.POINTER(Camera), i32, i32, vp, vp, vp, vp, vp, i32]
        lib.rtb_intersect_rays.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp]
        lib.rtb_query_rays.argtypes = [vp, vp, i64, vp, vp, C.c_float, i32, vp, vp, vp, vp, vp, vp]
        lib.rtb_query_points.argtypes = [vp, vp, i64, vp, vp, C.c_float, i32, vp, vp, vp, vp, vp, vp]
        lib.rtb_scene_mesh_moments.argtypes = [vp, vp, vp]
        lib.rtb_query_winding.argtypes = [vp, vp, i64, vp, C.c_float, vp, vp, vp]
        lib.rtb_query_triangles.argtypes = [vp, vp, i64, vp, i32, vp, vp, i64, vp, vp]
        lib.rtb_forget_schedule.argtypes = [vp]
        lib.rtb_device_alloc.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
        lib.rtb_device_free.argtypes = [vp, vp]
        lib.rtb_device_download.argtypes = [vp, vp, vp, C.c_size_t]
        lib.rtb_ipc_export.argtypes = [vp, vp, C.c_char_p]
        lib.rtb_ipc_open.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
        lib.rtb_ipc_close.argtypes = [vp, vp]
        lib.rtb_scatter_shard_device.argtypes = [vp, vp, vp, C.POINTER(Frame), vp]
        lib.rtb_multi_init.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(vp)]
        lib.rtb_multi_shutdown.argtypes = [vp]
        lib.rtb_multi_count.argtypes = [vp]
        lib.rtb_multi_ctx.argtypes = [vp, C.c_int]
        lib.rtb_multi_ctx.restype = vp
        lib.rtb_multi_last_error.argtypes = [vp]
        lib.rtb_multi_last_error.restype = C.c_char_p
        lib.rtb_multi_scene_upload.argtypes = [vp, C.POINTER(FlatScene), C.POINTER(vp)]
        lib.rtb_multi_scene_free.argtypes = [vp, vp]
        lib.rtb_multi_scene_upload_bytes.argtypes = [vp]
        lib.rtb_multi_scene_upload_bytes.restype = i64
        lib.rtb_multi_render.argtypes = [vp, vp, C.POINTER(Camera), C.POINTER(RenderSetting), C.POINTER(Frame), vp, C.POINTER(Stats)]
        lib.rtb_multi_scene_mesh_update.argtypes = [vp, vp, i32, vp, i64, i32]
        _cuda = lib
    return _cuda


def host_lib():
    global _host
    if _host is None:
        cuda_lib()
        if not os.path.exists(HOST_LIB):
            raise RtbError(f"{HOST_LIB} is missing: run `python __graft_entry__.py build`")
        lib = C.CDLL(HOST_LIB)
        vp = C.c_void_p
        lib.rtbh_preset_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_char_p]
        lib.rtbh_preset_create.restype = vp
        lib.rtbh_perf_scene_create.argtypes = [C.c_float, C.c_float, C.c_int, C.c_int, C.c_int]
        lib.rtbh_perf_scene_create.restype = vp
        lib.rtbh_free.argtypes = [vp]
        lib.rtbh_flat.argtypes = [vp]
        lib.rtbh_flat.restype = C.POINTER(FlatScene)
        lib.rtbh_camera.argtypes = [vp]
        lib.rtbh_camera.restype = C.POINTER(Camera)
        lib.rtbh_setting.argtypes = [vp]
        lib.rtbh_setting.restype = C.POINTER(RenderSetting)
        for f in ("rtbh_prepare_ms", "rtbh_build_ms"):
            getattr(lib, f).argtypes = [vp]
            getattr(lib, f).restype = C.c_double
        lib.rtbh_host_bytes.argtypes = [vp]
        lib.rtbh_host_bytes.restype = C.c_int64
        lib.rtbh_stats.argtypes = [vp, C.POINTER(C.c_int64)]
        for f in ("rtbh_tri_hash", "rtbh_struct_hash"):
            getattr(lib, f).argtypes = [vp]
            getattr(lib, f).restype = C.c_uint64
        lib.rtbh_script_run.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int,
                                        C.c_char_p, vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(Stats)]
        lib.rtbh_script_run_ex.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_int,
                                           C.c_char_p, vp, C.POINTER(C.c_int), C.POINTER(Stats), C.POINTER(C.c_int), C.c_char_p, C.c_int]
        lib.rtbh_script_run8.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int,
                                         C.c_char_p, vp, C.c_char_p, C.POINTER(C.c_int), C.POINTER(Stats)]
        lib.rtbh_perf_test.argtypes = [C.c_float, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp, vp, vp,
                                       C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]
        lib.rtbh_last_error.restype = C.c_char_p
        lib.rtbh_intersect_batch.argtypes = [vp, C.c_int64, vp, vp, vp, vp, vp]
        lib.rtbh_intersect_one.argtypes = [vp, vp, vp, vp, vp, vp]
        _host = lib
    return _host


def stl_fixture():
    return os.path.join(PKG, "assets", "ball.stl")  # the 528-triangle mesh of preset 3 (reference Scripts.cpp:113-168 reads ball.stl)


def _alg(a):
    return ALGORITHMS[a] if isinstance(a, str) else int(a)


def make_setting(name):
    return RenderSetting(*SETTINGS[name])


# ---- host side: preset scenes built by the C++ host API ----------------------------------------
class PresetScene:
    """A reference preset (Scripts.cpp Script1..5) built and flattened by the C++ host library."""

    def __init__(self, preset, algorithm="linear", segments=150, stl_path=None):
        lib = host_lib()
        self.preset, self.algorithm, self.segments = preset, algorithm, segments
        self._h = lib.rtbh_preset_create(preset, _alg(algorithm), segments, (stl_path or stl_fixture()).encode())
        if not self._h:
            raise RtbError("rtbh_preset_create failed (bad preset / algorithm / STL path)")
        self.flat = lib.rtbh_flat(self._h)
        self.camera = lib.rtbh_camera(self._h).contents
        self.setting = lib.rtbh_setting(self._h).contents

    def pin(self):
        """Page-lock the flat scene's arrays where they lie (rtb_host_register) and declare them page-locked and stable
        (rtb_flat_scene.arrays_page_locked): uploads then copy host -> device straight out of them.  An array that cannot be
        registered (it shares a page with one that is) stays pageable; the library stages such an array as before."""
        if getattr(self, "_pinned", None):
            return self
        lib = cuda_lib()
        self._pinned = [addr for addr, nbytes in self.flat.contents.arrays()
                        if nbytes >= (64 << 10) and lib.rtb_host_register(C.c_void_p(addr), C.c_size_t(nbytes)) == 0]
        self.flat.contents.arrays_page_locked = 1
        return self

    def unpin(self):
        for addr in getattr(self, "_pinned", None) or []:
            cuda_lib().rtb_host_unregister(C.c_void_p(addr))
        self._pinned = []
        if self._h:
            self.flat.contents.arrays_page_locked = 0

    def close(self):
        if self._h:
            self.unpin()
            host_lib().rtbh_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def prepare_ms(self):
        return host_lib().rtbh_prepare_ms(self._h)

    @property
    def build_ms(self):
        return host_lib().rtbh_build_ms(self._h)

    @property
    def host_bytes(self):
        return host_lib().rtbh_host_bytes(self._h)

    def stats(self):
        out = (C.c_int64 * 16)()
        host_lib().rtbh_stats(self._h, out)
        return {k: int(out[i]) for i, k in enumerate(STAT_NAMES)}

    def struct_hash(self):
        return int(host_lib().rtbh_struct_hash(self._h))

    def tri_hash(self):
        return int(host_lib().rtbh_tri_hash(self._h))

    def triangles(self):
        f = self.flat.contents
        n = f.n_tris
        if n == 0:
            return np.zeros((0, 12), np.float32), np.zeros(0, np.int32)
        tri = np.ctypeslib.as_array(f.tri, shape=(n, 12)).copy()
        mat = np.ctypeslib.as_array(f.tri_material, shape=(n,)).copy()
        return tri, (mat == mat[-1]).astype(np.int32)

    def intersect_batch(self, rays):
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 6)
        n = rays.shape[0]
        hid, ht = np.zeros(n, np.int32), np.zeros(n, np.float32)
        pos, nrm = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        rc = host_lib().rtbh_intersect_batch(self._h, n, rays.ctypes.data, hid.ctypes.data, ht.ctypes.data,
                                             pos.ctypes.data, nrm.ctypes.data)
        if rc != 0:
            raise RtbError("GeometrySet::intersectBatch failed: " + host_lib().rtbh_last_error().decode())
        return hid, ht, pos, nrm

    def intersect_one(self, ray):
        ray = np.ascontiguousarray(ray, np.float32).reshape(6)
        hid, ht = C.c_int32(-1), C.c_float(0)
        pos, nrm = np.zeros(3, np.float32), np.zeros(3, np.float32)
        host_lib().rtbh_intersect_one(self._h, ray.ctypes.data, C.byref(hid), C.byref(ht), pos.ctypes.data, nrm.ctypes.data)
        return hid.value, ht.value, pos, nrm


def set_exact_grid_binning(on):
    """Tunnels built from now on bin triangles into grid cells with the exact overlap test (reference
    Triangle.cpp:152-199, compiled out at Tunnel.cpp:435-445) instead of the bounding-box overlap."""
    host_lib().rtbh_set_exact_grid_binning(1 if on else 0)


def set_kd_on_device(on):
    """Tunnels built from now on leave a KdTreeSAH accelerator to the device builder of rtb_scene_upload."""
    host_lib().rtbh_set_kd_on_device(1 if on else 0)


def set_stl_as_mesh(on):
    """Preset 3 built from now on loads its STL as one triangle mesh (GeometrySet::addStlMesh, RTB_PRIM_MESH) instead of
    loose triangles: the same triangles and hit ids, traversed through a hierarchy built on the device."""
    host_lib().rtbh_set_stl_as_mesh(1 if on else 0)


def set_grid_on_device(on):
    """Tunnels built from now on leave RegularGrid / FlatGrid to the device builder of rtb_scene_upload."""
    host_lib().rtbh_set_grid_on_device(1 if on else 0)


class PerfScene(PresetScene):
    """The scene of the reference's PerformanceTest program (tunnel built by that program's own generator and
    k-d builder + the plane closing its exit), built and flattened by the C++ host library."""

    def __init__(self, radius=2000.0, angle=1.5708, arch_seg=150, path_seg=150, algorithm="sah"):
        lib = host_lib()
        self.preset, self.algorithm, self.segments = 0, algorithm, path_seg
        self._h = lib.rtbh_perf_scene_create(radius, angle, arch_seg, path_seg, _alg(algorithm))
        if not self._h:
            raise RtbError("rtbh_perf_scene_create failed (bad algorithm / tessellation)")
        self.flat = lib.rtbh_flat(self._h)
        self.camera = lib.rtbh_camera(self._h).contents
        self.setting = lib.rtbh_setting(self._h).contents


def script_run(preset, algorithm="linear", segments=150, width=400, height=300, samples=1, seed=0, device=0,
               stl_path=None):
    """The drop-in path: Script::Run(CudaRenderer::Render, ...) -- returns (image[y][x][3], info)."""
    lib = host_lib()
    rgb = np.zeros((width, height, 3), np.float32)
    prep, exe, st = C.c_int(0), C.c_int(0), Stats()
    rc = lib.rtbh_script_run(preset, _alg(algorithm), segments, width, height, samples, seed, device,
                             (stl_path or stl_fixture()).encode(), rgb.ctypes.data, C.byref(prep), C.byref(exe),
                             C.byref(st))
    if rc != 0:
        raise RtbError(f"Script::Run failed rc={rc}: {lib.rtbh_last_error().decode()}")
    info = st.as_dict()
    info.update(prepare_ms=prep.value, exec_ms=exe.value)
    return np.ascontiguousarray(rgb.transpose(1, 0, 2)), info


def script_run_ex(preset, algorithm="linear", segments=150, width=400, height=300, samples=1, seed=0, device=0, n_devices=1,
                  stl_path=None):
    """Script::Run(CudaRenderer::Render, ...) on n_devices GPUs with the reference's ProgressCallback and LogCallback attached;
    returns (image[y][x][3] or None, info) -- info carries rc, the progress calls seen and the log text."""
    lib = host_lib()
    rgb = np.zeros((width, height, 3), np.float32)
    exe, st, prog = C.c_int(0), Stats(), (C.c_int * 4)()
    log = C.create_string_buffer(4096)
    rc = lib.rtbh_script_run_ex(preset, _alg(algorithm), segments, width, height, samples, seed, device, n_devices,
                                (stl_path or stl_fixture()).encode(), rgb.ctypes.data, C.byref(exe), C.byref(st), prog, log, 4096)
    info = st.as_dict()
    info.update(rc=rc, exec_ms=exe.value, progress_calls=prog[0], progress_last=prog[1], progress_total=prog[2],
                progress_monotone=bool(prog[3]), log=log.value.decode(errors="replace"))
    return (np.ascontiguousarray(rgb.transpose(1, 0, 2)) if rc == 0 else None), info


def script_run8(preset, algorithm="linear", segments=150, width=400, height=300, samples=1, seed=0, device=0,
                stl_path=None, bmp_path=None):
    """Drop-in path with the reference's 8-bit output stage; returns (uint8 image[y][x][3], info)."""
    lib = host_lib()
    rgb = np.zeros((width, height, 3), np.uint8)
    exe, st = C.c_int(0), Stats()
    rc = lib.rtbh_script_run8(preset, _alg(algorithm), segments, width, height, samples, seed, device,
                              (stl_path or stl_fixture()).encode(), rgb.ctypes.data,
                              bmp_path.encode() if bmp_path else None, C.byref(exe), C.byref(st))
    if rc != 0:
        raise RtbError(f"Script::Run (8-bit) failed rc={rc}: {lib.rtbh_last_error().decode()}")
    info = st.as_dict()
    info.update(exec_ms=exe.value)
    return np.ascontiguousarray(rgb.transpose(1, 0, 2)), info


def perf_test(xy, radius=2000.0, angle=1.5708, arch_seg=150, path_seg=150, algorithm="sah", max_depth=200):
    """The reference's PerformanceTest console benchmark on the GPU (host C++: rt::PerformanceTest)."""
    xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
    n = xy.shape[0]
    out = {"reached": np.zeros(n, np.int32), "depth": np.zeros(n, np.int32), "last_id": np.zeros(n, np.int32),
           "last_pos": np.zeros((n, 3), np.float32)}
    total, b, pre, tr = C.c_int64(0), C.c_double(0), C.c_double(0), C.c_double(0)
    rc = host_lib().rtbh_perf_test(radius, angle, arch_seg, path_seg, _alg(algorithm), n, xy.ctypes.data, max_depth,
                                   out["reached"].ctypes.data, out["depth"].ctypes.data, out["last_id"].ctypes.data,
                                   out["last_pos"].ctypes.data, C.byref(total), C.byref(b), C.byref(pre), C.byref(tr))
    if rc != 0:
        raise RtbError(f"PerformanceTest failed rc={rc}: {host_lib().rtbh_last_error().decode()}")
    out.update(total_rays=total.value, build_ms=b.value, preprocess_ms=pre.value, trace_ms=tr.value)
    return out


# ---- device side: context + uploaded scene over the C ABI --------------------------------------
class Context:
    def __init__(self, device=0):
        self._lib = cuda_lib()
        self._h = C.c_void_p()
        rc = self._lib.rtb_init(device, C.byref(self._h))
        if rc != 0:
            raise RtbError(f"rtb_init({device}) failed rc={rc}: {self._lib.rtb_last_error(None).decode()}")
        self.device = device

    def close(self):
        if self._h:
            self._lib.rtb_shutdown(self._h)
            self._h = C.c_void_p()

    def _check(self, rc, what):
        if rc != 0:
            raise RtbError(f"{what} failed rc={rc}: {self._lib.rtb_last_error(self._h).decode()}")

    def upload(self, flat):
        return DeviceScene(self, flat)

    def forget_schedule(self):
        """The next frame runs like the first frame of a new view (raster order, no latency tiers)."""
        self._check(self._lib.rtb_forget_schedule(self._h), "rtb_forget_schedule")

    # ---- one frame buffer, several devices (RTB_LAYOUT_GLOBAL; include/rtb.h section A) ----
    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self._check(self._lib.rtb_device_alloc(self._h, nbytes, C.byref(p)), "rtb_device_alloc")
        return p.value

    def device_free(self, ptr):
        self._check(self._lib.rtb_device_free(self._h, C.c_void_p(ptr)), "rtb_device_free")

    def device_download(self, ptr, out):
        """synchronous copy of out.nbytes bytes of a device frame into the numpy array `out`"""
        self._check(self._lib.rtb_device_download(self._h, C.c_void_p(ptr), out.ctypes.data, out.nbytes), "rtb_device_download")
        return out

    def ipc_export(self, ptr):
        buf = C.create_string_buffer(IPC_HANDLE_BYTES)
        self._check(self._lib.rtb_ipc_export(self._h, C.c_void_p(ptr), buf), "rtb_ipc_export")
        return buf.raw

    def ipc_open(self, handle):
        p = C.c_void_p()
        self._check(self._lib.rtb_ipc_open(self._h, C.create_string_buffer(bytes(handle), IPC_HANDLE_BYTES), C.byref(p)), "rtb_ipc_open")
        return p.value

    def scatter_shard_device(self, local_ptr, frame_ptr, frame, stream=0):
        """rtb_scatter_shard_device: a rank's local shard image -> its place in the whole (possibly peer-mapped) frame."""
        self._check(self._lib.rtb_scatter_shard_device(self._h, C.c_void_p(local_ptr), C.c_void_p(frame_ptr), C.byref(frame), C.c_void_p(stream)),
                    "rtb_scatter_shard_device")

    def ipc_close(self, ptr):
        self._check(self._lib.rtb_ipc_close(self._h, C.c_void_p(ptr)), "rtb_ipc_close")


class MultiContext:
    """rtb_multi_*: one host thread drives n devices; rtb_multi_render returns ONE assembled host frame."""

    def __init__(self, n_devices, devices=None):
        self._lib = cuda_lib()
        self._h = C.c_void_p()
        arr = (C.c_int * n_devices)(*devices) if devices is not None else None
        rc = self._lib.rtb_multi_init(n_devices, arr, C.byref(self._h))
        if rc != 0:
            raise RtbError(f"rtb_multi_init({n_devices}) failed rc={rc}: {self._lib.rtb_last_error(None).decode()}")
        self.n = n_devices

    def close(self):
        if self._h:
            self._lib.rtb_multi_shutdown(self._h)
            self._h = C.c_void_p()

    def _check(self, rc, what):
        if rc != 0:
            raise RtbError(f"{what} failed rc={rc}: {self._lib.rtb_multi_last_error(self._h).decode()}")

    def upload(self, flat):
        return MultiScene(self, flat)


class MultiScene:
    def __init__(self, multi, flat):
        self.multi = multi
        self._h = C.c_void_p()
        multi._check(multi._lib.rtb_multi_scene_upload(multi._h, flat, C.byref(self._h)), "rtb_multi_scene_upload")

    def close(self):
        if self._h:
            self.multi._lib.rtb_multi_scene_free(self.multi._h, self._h)
            self._h = C.c_void_p()

    @property
    def upload_bytes(self):
        return int(self.multi._lib.rtb_multi_scene_upload_bytes(self._h))

    def mesh_update(self, records, mesh_index=0, refit=False):
        """rtb_multi_scene_mesh_update: DeviceScene.mesh_update on every device; `records` is a [count][12] float32 numpy array."""
        rec = _host_records(records)
        self.multi._check(self.multi._lib.rtb_multi_scene_mesh_update(self.multi._h, self._h, mesh_index, rec.ctypes.data, len(rec),
                                                                      MESH_REFIT if refit else MESH_REBUILD), "rtb_multi_scene_mesh_update")

    def render(self, camera, setting, frame, out=None):
        """The whole frame into ONE host buffer: [height][width][3] (reference order [width][height][3] with LAYOUT_REFERENCE)."""
        if out is None:
            shape = (frame.width, frame.height, 3) if frame.layout & LAYOUT_REFERENCE else (frame.height, frame.width, 3)
            if frame.layout & OUTPUT_MOMENTS:
                shape = shape[:2] + (6,)
            out = np.zeros(shape, np.uint8 if frame.layout & OUTPUT_RGB8 else np.float32)
        st = Stats()
        self.multi._check(self.multi._lib.rtb_multi_render(self.multi._h, self._h, C.byref(camera), C.byref(setting), C.byref(frame),
                                                           out.ctypes.data, C.byref(st)), "rtb_multi_render")
        return out, st.as_dict()


def unshard_device(ctx, gathered_ptr, image_ptr, width, height, world, row_block, rows_per_rank, stream=0):
    ctx._check(ctx._lib.rtb_unshard_device(ctx._h, C.c_void_p(gathered_ptr), C.c_void_p(image_ptr), width, height, world,
                                           row_block, rows_per_rank, C.c_void_p(stream)), "rtb_unshard_device")


def unshard_cols_device(ctx, gathered_ptr, image_ptr, width, height, world, row_block, col_block, stream=0):
    ctx._check(ctx._lib.rtb_unshard_cols_device(ctx._h, C.c_void_p(gathered_ptr), C.c_void_p(image_ptr), width, height, world,
                                                row_block, col_block, C.c_void_p(stream)), "rtb_unshard_cols_device")


def _host_records(records):
    return np.ascontiguousarray(records, np.float32).reshape(-1, 12)


class PinnedArray:
    """float32 numpy view over page-locked host memory from rtb_host_alloc."""

    def __init__(self, shape):
        self.shape = tuple(int(x) for x in shape)
        n = int(np.prod(self.shape))
        self._p = C.c_void_p()
        rc = cuda_lib().rtb_host_alloc(max(n, 1) * 4, C.byref(self._p))
        if rc != 0:
            raise RtbError("rtb_host_alloc failed: " + cuda_lib().rtb_last_error(None).decode())
        self.array = np.ctypeslib.as_array(C.cast(self._p, C.POINTER(C.c_float)), shape=(max(n, 1),))[:n].reshape(self.shape)

    def close(self):
        if self._p:
            cuda_lib().rtb_host_free(self._p)
            self._p = C.c_void_p()


def shard_rows(frame):
    return int(cuda_lib().rtb_shard_rows(C.byref(frame)))


def shard_width(frame):
    return int(cuda_lib().rtb_shard_width(C.byref(frame)))


def make_frame(width, height, samples=1, seed=0, rank=0, world=1, row_block=8, layout=LAYOUT_ROWMAJOR, counters=0, col_block=0,
               sample_first=0, sample_count=0):
    """col_block > 0 (and world > 1): column-block shard, local image [height][width / world] (include/rtb.h).
    sample_count > 0: Monte-Carlo sample shard [sample_first, sample_first + sample_count) of `samples`."""
    return Frame(width, height, samples, seed, rank, world, row_block, layout, counters, col_block, sample_first, sample_count)


def shard_col_indices(width, y, rank, world, row_block, col_block):
    """Global x of each local column of row y of a column-block shard: block row by = y // row_block owns the
    column blocks bx with (bx + by) % world == rank (mirror of localToGlobal in csrc/rtb_kernels.cuh)."""
    by = y // row_block
    shift = (rank - by) % world
    xs = []
    for c in range(width // (world * col_block)):
        bx = c * world + shift
        xs.extend(range(bx * col_block, (bx + 1) * col_block))
    return np.asarray(xs, np.int64)


def sample_shard(samples, rank, world):
    """(sample_first, sample_count) of rank's share of a Monte-Carlo frame's samples: contiguous ranges, the first
    samples % world ranks take one more (rtb_frame.sample_first / sample_count)."""
    base, extra = divmod(samples, world)
    first = rank * base + min(rank, extra)
    return first, base + (1 if rank < extra else 0)


def shard_pixel_mask(width, height, rank, world, row_block=8, col_block=0):
    """bool [height][width]: the pixels of the frame rank `rank` stores with RTB_LAYOUT_GLOBAL (mirror of localToGlobal
    in csrc/rtb_kernels.cuh: row blocks dealt round-robin, or column blocks rotated from block row to block row)."""
    m = np.zeros((height, width), bool)
    if col_block and world > 1:
        for y in range(height):
            m[y, shard_col_indices(width, y, rank, world, row_block, col_block)] = True
    else:
        m[shard_row_indices(height, rank, world, row_block)] = True
    return m


def shard_row_indices(height, rank, world, row_block=8):
    """Global y of each local row of a shard (block b of row_block rows goes to rank b % world)."""
    ys = []
    b = rank
    while b * row_block < height:
        ys.extend(range(b * row_block, min((b + 1) * row_block, height)))
        b += world
    return np.asarray(ys, np.int64)


class DeviceScene:
    def __init__(self, ctx, flat):
        self.ctx = ctx
        self._h = C.c_void_p()
        self._moments = False  # rtb_scene_mesh_moments has run (winding_numbers builds them on first use)
        ctx._check(ctx._lib.rtb_scene_upload(ctx._h, flat, C.byref(self._h)), "rtb_scene_upload")

    def close(self):
        if self._h:
            self.ctx._lib.rtb_scene_free(self.ctx._h, self._h)
            self._h = C.c_void_p()

    @property
    def device_bytes(self):
        return int(self.ctx._lib.rtb_scene_device_bytes(self._h))

    @property
    def upload_bytes(self):
        """bytes the upload copied from host memory (the packed / pair streams are produced on the device)"""
        return int(self.ctx._lib.rtb_scene_upload_bytes(self._h))

    def grid_hash(self):
        """(canonical structure hash, {dims, occupied cells, references, longest list}) of the grid on the device."""
        h, st = C.c_uint64(0), (C.c_int64 * 6)()
        self.ctx._check(self.ctx._lib.rtb_scene_grid_hash(self.ctx._h, self._h, C.byref(h), st), "rtb_scene_grid_hash")
        return int(h.value), dict(grid_x=st[0], grid_y=st[1], grid_z=st[2], cells_nonempty=st[3], cell_entries=st[4], cell_max=st[5])

    def kd_download(self):
        """(nodes [n][2] uint32, leaf_tris [m] uint32, levels, box) of the k-d tree resident on the device."""
        counts, box = (C.c_int64 * 3)(), (C.c_float * 6)()
        self.ctx._check(self.ctx._lib.rtb_scene_kd_download(self.ctx._h, self._h, None, 0, None, 0, counts, box), "rtb_scene_kd_download")
        nodes, refs = np.zeros((counts[0], 2), np.uint32), np.zeros(counts[1], np.uint32)
        self.ctx._check(self.ctx._lib.rtb_scene_kd_download(self.ctx._h, self._h, nodes.ctypes.data, counts[0], refs.ctypes.data, counts[1],
                                                            counts, box), "rtb_scene_kd_download")
        return nodes, refs, int(counts[2]), np.array(list(box), np.float32)

    def mesh_download(self, mesh_index=0):
        """(lo [n][2][3], hi [n][2][3] float32, child [n][2] int32, tri_order [m] uint32, depth) of the hierarchy of the
        mesh record `mesh_index` (include/rtb.h: rtb_bvhnode)."""
        counts = (C.c_int64 * 3)()
        lib = self.ctx._lib
        self.ctx._check(lib.rtb_scene_mesh_download(self.ctx._h, self._h, mesh_index, None, 0, None, 0, counts), "rtb_scene_mesh_download")
        nodes = (BvhNode * int(counts[0]))()
        order = np.zeros(counts[1], np.uint32)
        self.ctx._check(lib.rtb_scene_mesh_download(self.ctx._h, self._h, mesh_index, nodes, counts[0], order.ctypes.data, counts[1], counts),
                        "rtb_scene_mesh_download")
        raw = np.frombuffer(nodes, np.uint8).reshape(int(counts[0]), 64)
        f = raw[:, :48].copy().view(np.float32).reshape(-1, 12)
        child = raw[:, 48:56].copy().view(np.int32).reshape(-1, 2)
        return f[:, :6].reshape(-1, 2, 3), f[:, 6:].reshape(-1, 2, 3), child, order, int(counts[2])

    def mesh_update(self, records, mesh_index=0, refit=False, stream=None):
        """rtb_scene_mesh_update: replace the triangles of the mesh record `mesh_index` (include/rtb.h).  `records` is a
        [count][12] float32 numpy array (a, b, c, normal: the loose_tri format), or a contiguous CUDA float32 tensor on the
        context's device, read in place behind the work on `stream` (default: torch's current stream, its default stream
        included; an explicit 0 is the context's own stream).  refit=False
        rebuilds the hierarchy as an upload does; refit=True keeps its shape and recomputes its boxes."""
        flags = MESH_REFIT if refit else MESH_REBUILD
        if hasattr(records, "data_ptr"):  # a torch tensor
            import torch
            if not records.is_cuda or records.dtype != torch.float32 or not records.is_contiguous() or records.numel() % 12:
                raise RtbError("mesh_update: a tensor must be a contiguous CUDA float32 tensor of [count][12] records")
            if stream is None:
                stream = torch.cuda.current_stream(records.device).cuda_stream
                # torch's default stream has handle 0, which the library reads as its own stream (not ordered with the
                # legacy default stream): name the legacy stream instead
                stream = stream or CUDA_STREAM_LEGACY
            ptr, n = records.data_ptr(), records.numel() // 12
        else:
            rec = _host_records(records)
            ptr, n = rec.ctypes.data, len(rec)
        self.ctx._check(self.ctx._lib.rtb_scene_mesh_update(self.ctx._h, self._h, mesh_index, C.c_void_p(ptr), n, flags,
                                                            C.c_void_p(stream or 0)), "rtb_scene_mesh_update")

    def render(self, camera, setting, frame, out=None):
        """rtb_render with HOST buffers; returns (rows x width x 3 float32 | reference-order array, stats)."""
        rows = shard_rows(frame)
        if rows < 0:
            raise RtbError("bad frame: size / rank / world / row_block (must be a multiple of 8)")
        if out is None:
            shape = (frame.width, frame.height, 3) if frame.layout & LAYOUT_REFERENCE else (rows, shard_width(frame), 3)
            if frame.layout & OUTPUT_MOMENTS:
                shape = shape[:2] + (6,)
            out = np.zeros(shape, np.uint8 if frame.layout & OUTPUT_RGB8 else np.float32)
        st = Stats()
        self.ctx._check(self.ctx._lib.rtb_render(self.ctx._h, self._h, C.byref(camera), C.byref(setting), C.byref(frame),
                                                 out.ctypes.data, C.byref(st)), "rtb_render")
        return out, st.as_dict()

    def render_device(self, camera, setting, frame, device_ptr, stream=0, want_stats=False):
        """rtb_render_device into DEVICE memory (e.g. a torch tensor's data_ptr()) on `stream`."""
        st = Stats()
        self.ctx._check(self.ctx._lib.rtb_render_device(self.ctx._h, self._h, C.byref(camera), C.byref(setting),
                                                        C.byref(frame), C.c_void_p(device_ptr), C.c_void_p(stream),
                                                        C.byref(st) if want_stats else None), "rtb_render_device")
        return st.as_dict() if want_stats else None

    def trace_primary(self, camera, width, height, seq=True, seq_cap=0):
        n = width * height
        hid, ht = np.zeros(n, np.int32), np.zeros(n, np.float32)
        slen = np.zeros(n, np.int32) if seq else None
        shash = np.zeros(n, np.uint64) if seq else None
        sbuf = np.zeros((n, seq_cap), np.int32) if seq_cap else None
        p = lambda a: a.ctypes.data if a is not None else None
        self.ctx._check(self.ctx._lib.rtb_trace_primary(self.ctx._h, self._h, C.byref(camera), width, height, p(hid), p(ht),
                                                        p(slen), p(shash), p(sbuf), seq_cap), "rtb_trace_primary")
        return {"hit_id": hid, "hit_t": ht, "seq_len": slen, "seq_hash": shash, "seq_buf": sbuf}

    def intersect_rays(self, rays):
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 6)
        n = rays.shape[0]
        hid, ht = np.zeros(n, np.int32), np.zeros(n, np.float32)
        pos, nrm = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        self.ctx._check(self.ctx._lib.rtb_intersect_rays(self.ctx._h, self._h, n, rays.ctypes.data, hid.ctypes.data,
                                                         ht.ctypes.data, pos.ctypes.data, nrm.ctypes.data),
                        "rtb_intersect_rays")
        return hid, ht, pos, nrm

    def query(self, rays, tmax=None, any_hit=False, stream=None, out=None):
        """rtb_query_rays: closest hits under a strict per-ray distance bound, or occlusion (include/rtb.h), on the device and
        ordered on `stream` with no host synchronisation.  `rays` is a contiguous CUDA float32 tensor [n][6] (origin, direction)
        on the context's device; `tmax` None (no bound), a float, or a contiguous CUDA float32 tensor [n].  `stream` as in
        mesh_update: torch's current stream by default.  The outputs are allocated on that stream, or taken from `out`:
        closest: (hit_id int32 [n], hit_t float32 [n], position float32 [n][3], normal float32 [n][3]), any of them may be
        None; any_hit: a torch.bool tensor [n] (True: something lies on the ray before tmax)."""
        return self._device_query(self.ctx._lib.rtb_query_rays, "query", rays, 6, "rays", tmax, "tmax", any_hit, stream, out,
                                  "hit_id, hit_t, position, normal")

    def closest_points(self, points, max_dist=None, any_hit=False, stream=None, out=None):
        """rtb_query_points: the nearest point on the scene's TRIANGLES and MESH records within a strict per-point radius, or
        whether one lies within it (include/rtb.h), on the device and ordered on `stream` with no host synchronisation.
        `points` is a contiguous CUDA float32 tensor [n][3] on the context's device; `max_dist` None (no bound), a float, or a
        contiguous CUDA float32 tensor [n].  Streams and outputs as in query: closest: (hit_id int32 [n], distance float32 [n],
        position float32 [n][3], normal float32 [n][3]); any_hit: a torch.bool tensor [n] (True: a triangle lies within
        max_dist)."""
        return self._device_query(self.ctx._lib.rtb_query_points, "closest_points", points, 3, "points", max_dist, "max_dist",
                                  any_hit, stream, out, "hit_id, distance, position, normal")

    def _device_query(self, fn, what, inp, width, inp_name, bound_arg, bound_name, any_hit, stream, out, out_names):
        import torch
        dev = torch.device("cuda", self.ctx.device)
        if not (isinstance(inp, torch.Tensor) and inp.device == dev and inp.dtype == torch.float32 and inp.is_contiguous()
                and inp.dim() == 2 and inp.shape[1] == width):
            raise RtbError(f"{what}: {inp_name} must be a contiguous float32 tensor [n][{width}] on {dev}")
        n = inp.shape[0]
        bound, bound_all = None, float("inf")
        if isinstance(bound_arg, torch.Tensor):
            if bound_arg.device != dev or bound_arg.dtype != torch.float32 or not bound_arg.is_contiguous() or tuple(bound_arg.shape) != (n,):
                raise RtbError(f"{what}: a {bound_name} tensor must be a contiguous float32 tensor [n] on {dev}")
            bound = bound_arg
        elif bound_arg is not None:
            bound_all = float(bound_arg)
        stream, alloc_stream = _query_stream(dev, stream)
        specs = [((n,), torch.bool)] if any_hit else [((n,), torch.int32), ((n,), torch.float32), ((n, 3), torch.float32),
                                                     ((n, 3), torch.float32)]
        if n == 0 and out is None:
            return torch.zeros(0, dtype=torch.bool, device=dev) if any_hit else \
                tuple(torch.zeros(shape, dtype=dt, device=dev) for shape, dt in specs)
        if out is None:
            with torch.cuda.stream(alloc_stream):
                outs = [torch.empty(shape, dtype=dt, device=dev) for shape, dt in specs]
        else:
            outs = [out] if any_hit else list(out)
            if len(outs) != len(specs) or (any_hit and outs[0] is None):
                raise RtbError(f"{what}: out must be a bool tensor (any_hit) or a 4-tuple ({out_names})")
            for o, (shape, dt) in zip(outs, specs):
                if o is not None and (not isinstance(o, torch.Tensor) or o.device != dev or o.dtype != dt or
                                      tuple(o.shape) != shape or not o.is_contiguous()):
                    raise RtbError(f"{what}: an output must be a contiguous {dt} tensor {list(shape)} on {dev}")
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        args = [None, None, None, None, p(outs[0])] if any_hit else [p(o) for o in outs] + [None]
        self.ctx._check(fn(self.ctx._h, self._h, n, p(inp), p(bound), bound_all, QUERY_ANY if any_hit else QUERY_CLOSEST, *args,
                           C.c_void_p(stream or 0)), fn.__name__)
        return outs[0] if any_hit else tuple(outs)

    def mesh_moments(self, stream=None):
        """rtb_scene_mesh_moments: build the first-order moments of every mesh hierarchy (include/rtb.h), which winding
        queries on a scene with MESH records need; winding_numbers, contains and signed_distance call it on first use.
        `stream` as in mesh_update (torch's current stream by default).  A second call does nothing."""
        if self._moments:
            return
        if stream is None:
            import torch
            stream = torch.cuda.current_stream(torch.device("cuda", self.ctx.device)).cuda_stream or CUDA_STREAM_LEGACY
        self.ctx._check(self.ctx._lib.rtb_scene_mesh_moments(self.ctx._h, self._h, C.c_void_p(stream or 0)), "rtb_scene_mesh_moments")
        self._moments = True

    def winding_numbers(self, points, beta=2.0, stream=None, out=None):
        """rtb_query_winding: the generalised winding number of every point with respect to the scene's TRIANGLES and MESH
        records (include/rtb.h), on the device and ordered on `stream` with no host synchronisation: about 1 inside and 0
        outside a closed, outward-oriented surface.  `points` is a contiguous CUDA float32 tensor [n][3] on the context's
        device; beta >= 1 trades accuracy for speed on meshes (+inf: exact).  Streams and `out` (a float32 tensor [n]) as in
        query.  The first call builds the mesh moments (mesh_moments) on the same stream."""
        return self._winding(points, beta, stream, out, False)

    def contains(self, points, beta=2.0, stream=None, out=None):
        """rtb_query_winding's inside test: a torch.bool tensor [n], True where winding_numbers(points, beta) > 0.5."""
        return self._winding(points, beta, stream, out, True)

    def signed_distance(self, points, max_dist=None, beta=2.0, stream=None):
        """closest_points with the sign of contains: (signed distance float32 [n], hit_id, position, normal).  The distance is
        closest_points' distance, negated where contains(points, beta) is True; a point with no triangle within max_dist gets
        -inf inside and +inf outside.  Two launches on one stream, combined by torch elementwise ops on that stream."""
        import torch
        dev = torch.device("cuda", self.ctx.device)
        stream, alloc_stream = _query_stream(dev, stream)
        hit_id, dist, pos, nrm = self.closest_points(points, max_dist, stream=stream)
        ins = self.contains(points, beta, stream=stream)
        with torch.cuda.stream(alloc_stream):
            sd = torch.where(hit_id >= 0, dist, float("inf"))
            sd = torch.where(ins, -sd, sd)
        return sd, hit_id, pos, nrm

    def _winding(self, points, beta, stream, out, inside):
        import torch
        dev = torch.device("cuda", self.ctx.device)
        what = "contains" if inside else "winding_numbers"
        if not (isinstance(points, torch.Tensor) and points.device == dev and points.dtype == torch.float32 and points.is_contiguous()
                and points.dim() == 2 and points.shape[1] == 3):
            raise RtbError(f"{what}: points must be a contiguous float32 tensor [n][3] on {dev}")
        n = points.shape[0]
        stream, alloc_stream = _query_stream(dev, stream)
        dt = torch.bool if inside else torch.float32
        if out is None:
            with torch.cuda.stream(alloc_stream):
                out = torch.empty(n, dtype=dt, device=dev)
        elif not (isinstance(out, torch.Tensor) and out.device == dev and out.dtype == dt and tuple(out.shape) == (n,) and out.is_contiguous()):
            raise RtbError(f"{what}: out must be a contiguous {dt} tensor [{n}] on {dev}")
        if n == 0:
            return out
        self.mesh_moments(stream)
        p = C.c_void_p(out.data_ptr())
        self.ctx._check(self.ctx._lib.rtb_query_winding(self.ctx._h, self._h, n, C.c_void_p(points.data_ptr()), float(beta),
                                                        None if inside else p, p if inside else None, C.c_void_p(stream or 0)),
                        "rtb_query_winding")
        return out

    def intersects(self, tris, stream=None, out=None):
        """rtb_query_triangles with QUERY_ANY: a torch.bool tensor [m], True where the query triangle shares a point with one
        of the scene's TRIANGLES or MESH triangles, decided exactly (include/rtb.h; degenerate triangles never intersect).
        `tris` is a contiguous CUDA float32 tensor [m][12] (a, b, c, normal; the normal is ignored) on the context's device.
        On the device and ordered on `stream` with no host synchronisation; streams and `out` (a bool tensor [m]) as in
        query."""
        import torch
        tris, dev = self._query_tris(tris, "intersects")
        m = tris.shape[0]
        stream, alloc_stream = _query_stream(dev, stream)
        if out is None:
            with torch.cuda.stream(alloc_stream):
                out = torch.empty(m, dtype=torch.bool, device=dev)
        elif not (isinstance(out, torch.Tensor) and out.device == dev and out.dtype == torch.bool and tuple(out.shape) == (m,)
                  and out.is_contiguous()):
            raise RtbError(f"intersects: out must be a contiguous bool tensor [{m}] on {dev}")
        if m == 0:
            return out
        self.ctx._check(self.ctx._lib.rtb_query_triangles(self.ctx._h, self._h, m, C.c_void_p(tris.data_ptr()), QUERY_ANY,
                                                          C.c_void_p(out.data_ptr()), None, 0, None, C.c_void_p(stream or 0)),
                        "rtb_query_triangles")
        return out

    def intersecting_pairs(self, tris, capacity=None, stream=None):
        """rtb_query_triangles with QUERY_PAIRS: an int64 tensor [P][2] of every (i, hit_id) whose triangles share a point,
        sorted lexicographically.  `tris` as in intersects.  This reads the pair count back, so it SYNCHRONISES with
        `stream`; the query runs a second time only when the first buffer of `capacity` pairs (default: m) was too small."""
        import torch
        tris, dev = self._query_tris(tris, "intersecting_pairs")
        m = tris.shape[0]
        stream, alloc_stream = _query_stream(dev, stream)
        cap = m if capacity is None else int(capacity)
        if cap < 0:
            raise RtbError("intersecting_pairs: capacity must be >= 0")
        with torch.cuda.stream(alloc_stream):
            count = torch.empty(1, dtype=torch.int64, device=dev)
        while True:
            with torch.cuda.stream(alloc_stream):
                pairs = torch.empty((cap, 2), dtype=torch.int32, device=dev)
            self.ctx._check(self.ctx._lib.rtb_query_triangles(self.ctx._h, self._h, m, C.c_void_p(tris.data_ptr()), QUERY_PAIRS,
                                                              None, C.c_void_p(pairs.data_ptr()) if cap else None, cap,
                                                              C.c_void_p(count.data_ptr()), C.c_void_p(stream or 0)),
                            "rtb_query_triangles")
            alloc_stream.synchronize()
            total = int(count.cpu()[0])
            if total <= cap:
                break
            cap = total
        with torch.cuda.stream(alloc_stream):
            p = pairs[:total].to(torch.int64)
            p = p[torch.argsort(p[:, 0] * (1 << 32) + p[:, 1])]
        alloc_stream.synchronize()
        return p

    def _query_tris(self, tris, what):
        import torch
        dev = torch.device("cuda", self.ctx.device)
        if not (isinstance(tris, torch.Tensor) and tris.device == dev and tris.dtype == torch.float32 and tris.is_contiguous()
                and tris.dim() == 2 and tris.shape[1] == 12):
            raise RtbError(f"{what}: tris must be a contiguous float32 tensor [m][12] on {dev}")
        return tris, dev


def _query_stream(dev, stream):
    """(handle, torch stream) of a query: torch's current stream by default (cudaStreamLegacy for its default stream: see
    DeviceScene.mesh_update); the torch stream is the one outputs are allocated on."""
    import torch
    if stream is None:
        stream = torch.cuda.current_stream(dev).cuda_stream or CUDA_STREAM_LEGACY
    alloc_stream = torch.cuda.ExternalStream(stream, device=dev) if stream not in (0, CUDA_STREAM_LEGACY) else \
        (torch.cuda.default_stream(dev) if stream == CUDA_STREAM_LEGACY else torch.cuda.current_stream(dev))
    return stream, alloc_stream


# ---- synthetic models -------------------------------------------------------------------------
def torus_triangles(n_triangles, seed=0, major=15.0, minor=6.0, center=(0.0, 16.0, 0.0)):
    """[n][12] float32 facets (normal, a, b, c: the binary STL facet order) of a closed torus tessellated into about
    n_triangles triangles (2 per grid quad, ring:tube = 2:1), every grid vertex displaced by a seeded jitter of 2 % of
    the tube's grid spacing.  Default size and place: inside the smallpt box of preset 3 once its STL offset is added."""
    nv = max(3, int(round(np.sqrt(n_triangles / 4.0))))
    nu = max(3, int(round(n_triangles / (2.0 * nv))))
    rng = np.random.default_rng(seed)
    u = (np.arange(nu) / nu * 2 * np.pi)[:, None]
    v = (np.arange(nv) / nv * 2 * np.pi)[None, :]
    rr = minor * (1 + 0.02 * (2 * np.pi / nv) * rng.uniform(-1, 1, (nu, nv)))
    x = (major + rr * np.cos(v)) * np.cos(u) + center[0]
    y = rr * np.sin(v) + center[1]
    z = (major + rr * np.cos(v)) * np.sin(u) + center[2]
    p = np.stack([x, y, z], -1).astype(np.float32)
    i, j = np.meshgrid(np.arange(nu), np.arange(nv), indexing="ij")
    i1, j1 = (i + 1) % nu, (j + 1) % nv
    a, b, c, d = p[i, j], p[i1, j], p[i1, j1], p[i, j1]
    t = np.concatenate([np.stack([a, b, c], -2).reshape(-1, 3, 3), np.stack([a, c, d], -2).reshape(-1, 3, 3)])
    n = np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0])
    n /= np.maximum(np.linalg.norm(n, axis=1, keepdims=True), 1e-30)
    return np.concatenate([n.astype(np.float32), t.reshape(-1, 9)], 1).astype(np.float32)


def write_stl(path, facets):
    """Binary STL of [n][12] float32 facets (normal, a, b, c), the format GeometrySet::addStlFile / addStlMesh read."""
    facets = np.ascontiguousarray(facets, np.float32).reshape(-1, 12)
    rec = np.zeros(len(facets), np.dtype([("f", "<f4", 12), ("attr", "<u2")]))
    rec["f"] = facets
    with open(path, "wb") as fh:
        fh.write(b"\0" * 80)
        fh.write(np.uint32(len(facets)).tobytes())
        fh.write(rec.tobytes())
