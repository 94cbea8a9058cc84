"""In-tree build of the two shared libraries of the package (no JIT cache, no pip install):

  librtb200.so       csrc/rtb_abi.cu  -- CUDA kernels + the C ABI of include/rtb.h   (nvcc, sm_100a)
  librtb200_host.so  host/rt_*.cpp    -- reference-shaped C++ host API + builders   (g++)

Parity flags: device code is compiled with -fmad=false (no FMA contraction) and the default
IEEE division / square root; host code with -ffp-contract=off and no fast-math, so the host
builders and the kernels evaluate the reference's float expressions as the x86-64 reference does.
"""
import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CUDA_LIB = os.path.join(PKG, os.environ.get("RTB_CUDA_LIB_NAME", "librtb200.so"))  # RTB_CUDA_LIB_NAME: experiment builds next to the product
HOST_LIB = os.path.join(PKG, "librtb200_host.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-fmad=false", "-Xcompiler", "-fPIC"]
# one translation unit per kernel family (the kernels are templates over probe x accelerator family x fold-stack size):
# compiled side by side, linked into one library
CUDA_UNITS = ["rtb_abi.cu", "rtb_k_chain.cu", "rtb_k_sm.cu", "rtb_k_oct.cu", "rtb_k_wide.cu", "rtb_k_mc.cu"]
CUDA_HEADERS = ["rtb_launch.h", "rtb_misc.cuh", "rtb_chain_sm.cuh", "rtb_chain_wide.cuh", "rtb_chain_oct.cuh", "rtb_build_grid.cuh",
                "rtb_kernels.cuh", "rtb_device.cuh", "rtb_pretest.h", "rtb_sat.h", "rtb_bvh.h", "rtb_build_bvh.cuh", "rtb_closest.h",
                "rtb_winding.h", "rtb_tritri.h"]
GXX_FLAGS = ["-O2", "-std=c++17", "-fopenmp", "-ffp-contract=off", "-fPIC", "-shared", "-Wall"]


def _newer(target, sources):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def build_cuda(force=False, verbose=False):
    from concurrent.futures import ThreadPoolExecutor
    csrc = os.path.join(PKG, "csrc")
    units = [os.path.join(csrc, f) for f in CUDA_UNITS]
    deps = units + [os.path.join(csrc, f) for f in CUDA_HEADERS] + [os.path.join(ROOT, "include", "rtb.h")]
    if not force and _newer(CUDA_LIB, deps):
        return CUDA_LIB
    extra = os.environ.get("RTB_NVCC_EXTRA", "").split()  # tuning experiments, e.g. -DRTB_CHAIN_MIN_CTAS=6
    objdir = os.path.join(PKG, "build" + ("_" + os.environ["RTB_CUDA_LIB_NAME"] if "RTB_CUDA_LIB_NAME" in os.environ else ""))
    os.makedirs(objdir, exist_ok=True)
    headers_t = max(os.path.getmtime(d) for d in deps[len(units):])

    def compile_unit(src):
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        if not force and not extra and os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(src), headers_t):
            return obj
        cmd = [_nvcc()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
        subprocess.check_call(cmd, cwd=PKG)
        return obj

    with ThreadPoolExecutor(max_workers=len(units)) as pool:
        objs = list(pool.map(compile_unit, units))
    subprocess.check_call([_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", CUDA_LIB] + objs, cwd=PKG)
    return CUDA_LIB


def build_host(force=False):
    src = [os.path.join(PKG, "host", f) for f in ("rt_scene.cpp", "rt_tunnel.cpp", "rt_render.cpp")]
    deps = src + [os.path.join(PKG, "host", "rt.h"), os.path.join(PKG, "csrc", "rtb_sat.h"), os.path.join(ROOT, "include", "rtb.h")]
    if not force and _newer(HOST_LIB, deps) and os.path.getmtime(HOST_LIB) >= os.path.getmtime(CUDA_LIB):
        return HOST_LIB
    # plain `g++` from PATH: the image's $CXX wrapper lacks libgomp
    cmd = ["g++"] + GXX_FLAGS + ["-o", HOST_LIB] + src + ["-L" + PKG, "-lrtb200", "-Wl,-rpath,$ORIGIN"]
    subprocess.check_call(cmd, cwd=PKG)
    return HOST_LIB


def build_all(force=False, verbose=False):
    build_cuda(force, verbose)
    build_host(force)
    return CUDA_LIB, HOST_LIB


if __name__ == "__main__":
    import sys
    build_all(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(CUDA_LIB)
    print(HOST_LIB)
