"""build.py -- compiles the library in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python waifu2x-converter-cpp_b200/build.py [--force]

Outputs (git-ignored, but they travel to the GPU box with a gpurun snapshot):
    waifu2x-converter-cpp_b200/libw2x_b200.so      the C-ABI product library (include/w2x_b200.h)
    waifu2x-converter-cpp_b200/w2x-converter       the drop-in CLI (host/main.cpp), if present
    waifu2x-converter-cpp_b200/w2x-bench-host      times w2xc::convertWithModels through host/w2xc.hpp (bench.py's e2e_cpp leg)
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libw2x_b200.so")
CLI = os.path.join(HERE, "w2x-converter")
BENCH_HOST = os.path.join(HERE, "w2x-bench-host")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-I", os.path.join(ROOT, "include"), "-I", CSRC,
          "-Xcompiler", "-fPIC,-fvisibility=hidden,-Wall,-Wextra"] + os.environ.get("W2X_BUILD_DEFS", "").split()
LIB_SOURCES = ["model.cpp", "geometry.cpp", "kernels_fp32.cu", "kernels_tc.cu", "image.cu", "engine.cu", "engine_band.cu",
               "engine_image.cu"]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _headers():
    hs = [os.path.join(ROOT, "include", "w2x_b200.h")]
    for d in (CSRC, os.path.join(HERE, "host")):
        if os.path.isdir(d):
            hs += [os.path.join(d, f) for f in os.listdir(d) if f.endswith((".h", ".hpp", ".cuh"))]
    return hs


def _compile(src, force):
    obj = os.path.join(OBJ, os.path.basename(src) + ".o")
    if force or _newer(obj, [src] + _headers()):
        cmd = [NVCC] + ARCH + COMMON + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
    return obj


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    srcs = [os.path.join(CSRC, s) for s in LIB_SOURCES]
    with cf.ThreadPoolExecutor(max_workers=len(srcs)) as ex:
        objs = list(ex.map(lambda s: _compile(s, force), srcs))
    if force or _newer(LIB, objs):
        cmd = [NVCC] + ARCH + ["-shared", "-o", LIB] + objs + ["-cudart", "static", "-Xlinker", "-z,defs", "-lpthread", "-ldl", "-lrt"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    main_cpp = os.path.join(HERE, "host", "main.cpp")
    if os.path.exists(main_cpp) and (force or _newer(CLI, [main_cpp, LIB] + _headers())):
        cmd = ["g++", "-O3", "-std=c++17", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(HERE, "host"),
               main_cpp, "-o", CLI, "-L", HERE, "-lw2x_b200", "-lz", "-pthread", "-Wl,-rpath,$ORIGIN"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"CLI build failed:\n{r.stdout}\n{r.stderr}")
    bench_cpp = os.path.join(HERE, "host", "bench_host.cpp")
    if os.path.exists(bench_cpp) and (force or _newer(BENCH_HOST, [bench_cpp, LIB] + _headers())):
        cmd = ["g++", "-O3", "-std=c++17", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(HERE, "host"),
               bench_cpp, "-o", BENCH_HOST, "-L", HERE, "-lw2x_b200", "-pthread", "-Wl,-rpath,$ORIGIN"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"bench host build failed:\n{r.stdout}\n{r.stderr}")
    if verbose:
        print("built", LIB)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
