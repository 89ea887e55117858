"""Whole images on the device (w2x_image_*, csrc/image.cu): the plumbing kernels restate host/imgproc.hpp with the same
fp32/fp64 operations in the same order and no contraction, so their results are bit-identical to the host path.  These
checks need no GPU: the shared arithmetic (csrc/image_math.h) against imgproc.hpp on the host, the compiled kernels'
SASS, and the entry points' argument checks."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT

PKG = os.path.join(ROOT, "waifu2x-converter-cpp_b200")
IMAGE_KERNELS = ("k_bgr8_to_yuv", "k_yuv_to_bgr8", "k_resize_nearest", "k_resizeILi4E", "k_resizeILi2E")


def build_driver(out):
    """tests/cpp/image_plumbing.cpp, compiled like the CLI (g++ -O3, no -march: no FMA on the host side)."""
    subprocess.check_call(["g++", "-O3", "-std=c++17", "-Wall", "-Wextra", "-I", os.path.join(PKG, "csrc"), "-I", os.path.join(PKG, "host"),
                           os.path.join(ROOT, "tests", "cpp", "image_plumbing.cpp"), "-o", out, "-pthread"])
    return out


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    return build_driver(str(tmp_path_factory.mktemp("cpp") / "image_plumbing"))


def test_device_arithmetic_is_bitwise_the_host_plumbing(driver):
    """image_math.h (host flavour, the kernels' loops) against imgproc.hpp on random 8-bit images and random fp32 YUV images
    with out-of-range values, NaN, +-0 and +-inf: colour conversion, nearest 2x, bicubic 2x, bilinear shrinks (ratios 3, 1.5,
    2.5, 0.5 through main.cpp's size arithmetic) and the 8-bit conversion, at 1x1, 2x3, 37x29, 45x33 and 640x400."""
    r = subprocess.run([driver, "selftest"], capture_output=True, text=True)
    assert r.returncode == 0 and "ALL OK" in r.stdout, r.stdout + r.stderr


def _sass_functions(lib_path):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    text = subprocess.check_output([exe, "-sass", lib_path], text=True)
    funcs, arch = {}, None
    for block in re.split(r"\n(?=arch = |\t\tFunction : )", text):
        m = re.match(r"arch = (\w+)", block)
        if m:
            arch = m.group(1)
            continue
        m = re.match(r"\t\tFunction : (\S+)", block)
        if m:
            funcs[m.group(1)] = (arch, block)
    return funcs


def test_image_kernels_are_sm100a_without_fma(w2x):
    funcs = _sass_functions(w2x.lib_path())
    for k in IMAGE_KERNELS:
        hits = [(name, arch, body) for name, (arch, body) in funcs.items() if k in name]
        assert hits, f"{k} not in the library's SASS"
        for name, arch, body in hits:
            assert arch == "sm_100a", (name, arch)
            ops = re.findall(r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)", body)
            assert ops, name
            contracted = sorted({o for o in ops if o.split(".")[0] in ("FFMA", "FFMA2", "DFMA", "HFMA2")})
            assert not contracted, (name, contracted)
            assert any(o.startswith("FMUL") for o in ops) or "nearest" in name, name   # the arithmetic is there, unfused


def test_image_entry_points_fail_with_a_status_without_a_context(w2x):
    L = w2x.lib()
    px = np.zeros((4, 5, 3), np.uint8)
    out = C.c_void_p()
    ptr = C.c_void_p(px.ctypes.data)
    assert L.w2x_image_create(None, ptr, 5, 4, 15, C.byref(out)) == 1 and not out.value
    assert "NULL context" in L.w2x_last_error().decode()
    assert L.w2x_image_create_device(None, ptr, 5, 4, 15, C.byref(out)) == 1 and not out.value
    assert L.w2x_image_create(None, ptr, 5, 4, 15, None) == 1
    L.w2x_image_destroy(None)
    w, h = C.c_int(-1), C.c_int(-1)
    assert L.w2x_image_size(None, C.byref(w), C.byref(h)) == 1 and w.value == -1
    for call in (lambda: L.w2x_image_denoise(None, None), lambda: L.w2x_image_scale2x(None, None),
                 lambda: L.w2x_image_resize_linear(None, 8, 8), lambda: L.w2x_image_download(None, ptr, 15),
                 lambda: L.w2x_image_download_device(None, ptr, 15), lambda: L.w2x_image_planes(None, ptr, ptr, ptr, 20)):
        assert call() == 1
        assert "NULL image" in L.w2x_last_error().decode()
