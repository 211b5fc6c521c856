"""In-tree build of the native libraries (no JIT cache: the .so files travel with the repo snapshot).

  _build/librt1w.so       the product: C ABI of include/rt1w.h + sm_100a kernels (nvcc, static cudart)
  _build/librt1w_host.so  the C++ mirror of the reference's scene API and scene functions (g++)
  _build/rt1w_main        demo driver mirroring the reference's `main` (PPM to stdout)

Run as `python raytracing-1w_b200/build.py [--force]`.
"""
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
OUT = os.path.join(PKG, "_build")

NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else (shutil.which("g++") or "g++")

CUDA_SRCS = ["csrc/api.cu", "csrc/render.cu", "csrc/denoise.cu", "csrc/lbvh.cu", "csrc/lower.cpp", "csrc/bvh.cpp", "csrc/bvh8.cpp"]
CUDA_HDRS = ["csrc/device_types.h", "csrc/flat_plans.h", "csrc/kernels.cuh", "csrc/render.h", "csrc/lower.h", "csrc/bvh.h", "csrc/bvh8.h", "csrc/nccl_dl.h", "csrc/lbvh.h", "csrc/philox.h", "../include/rt1w.h"]
HOST_SRCS = ["host/scenes.cpp", "host/host_api.cpp"]
HOST_HDRS = ["host/rt1w.hpp", "host/scenes.hpp", "host/host_api.h", "../include/rt1w.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    # f32 division and square root (shading, pdfs, f32 screens: never the f64 intersection solve) as MUFU + multiply
    # (2 ulp) instead of the IEEE sequences with their slow-path calls: the wave kernels are bound by their
    # instruction-cache footprint (DESIGN.md section 7)
    "-prec-div=false", "-prec-sqrt=false",
    "-Xcompiler", "-fPIC,-O3,-Wall", "-cudart", "static", "--shared", "-ccbin", GXX,
]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def _run(cmd):
    print("+", " ".join(cmd), flush=True)
    subprocess.check_call(cmd, cwd=PKG)


def build_product(force=False, extra_flags=(), variant=None):
    """variant: builds _build/variant_<variant>.so with extra -D flags (tuning sweeps; select with RT1W_LIB)."""
    os.makedirs(OUT, exist_ok=True)
    target = os.path.join(OUT, "librt1w.so" if not variant else f"variant_{variant}.so")
    deps = [os.path.join(PKG, p) for p in CUDA_SRCS + CUDA_HDRS] + [os.path.abspath(__file__)]
    if force or _stale(target, deps):
        _run([NVCC] + NVCC_FLAGS + list(extra_flags) + ["-o", target] + CUDA_SRCS)
    return target


def build_host(force=False):
    os.makedirs(OUT, exist_ok=True)
    target = os.path.join(OUT, "librt1w_host.so")
    deps = [os.path.join(PKG, p) for p in HOST_SRCS + HOST_HDRS]
    if force or _stale(target, deps):
        _run([GXX, "-O2", "-std=c++17", "-fPIC", "-Wall", "-shared", "-o", target] + HOST_SRCS)
    main_t = os.path.join(OUT, "rt1w_main")
    main_src = os.path.join(PKG, "host/main.cpp")
    if os.path.exists(main_src) and (force or _stale(main_t, deps + [main_src, os.path.join(OUT, "librt1w.so")])):
        _run([GXX, "-O2", "-std=c++17", "-Wall", "-o", main_t, "host/main.cpp"] + HOST_SRCS +
             ["-L" + OUT, "-lrt1w", "-Wl,-rpath,$ORIGIN"])
    return target


def build_oracle(force=False):
    odir = os.path.join(ROOT, "oracle")
    if force:
        subprocess.check_call(["make", "-C", odir, "clean"])
    subprocess.check_call(["make", "-C", odir])
    return os.path.join(odir, "_build", "liboracle.so")


def build_all(force=False):
    build_product(force)
    build_host(force)
    build_oracle(force)


if __name__ == "__main__":
    if "--variant" in sys.argv:  # python build.py --variant NAME -DRT1W_X=1 ...
        i = sys.argv.index("--variant")
        build_product(True, [a for a in sys.argv[i + 2:]], variant=sys.argv[i + 1])
    else:
        build_all("--force" in sys.argv)
