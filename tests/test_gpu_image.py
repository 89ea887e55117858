"""Whole images on the GPU (w2x_image_*, w2xc::DeviceImage, the CLI's device path): every stage bitwise equal to the host
plumbing of host/imgproc.hpp around w2x_convert_plane on the same context."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from test_image_plumbing import build_driver

PKG = os.path.join(ROOT, "waifu2x-converter-cpp_b200")
CLI = os.path.join(PKG, "w2x-converter")
SIZES = [(1, 1), (2, 3), (37, 29), (45, 33), (640, 400), (513, 768), (1920, 1080)]


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    return build_driver(str(tmp_path_factory.mktemp("cpp") / "image_plumbing"))


@pytest.fixture(scope="module")
def models(w2x, oracle_models):
    return {n: w2x.Model.from_arrays(om.weights, om.biases) for n, om in oracle_models.items()}


class Host:
    """The host side of every stage, from tests/cpp/image_plumbing.cpp (imgproc.hpp as host/main.cpp calls it)."""

    def __init__(self, exe, d):
        self.exe, self.d = exe, d

    def _run(self, *args):
        subprocess.check_call([self.exe, *map(str, args)])

    def yuv(self, bgr):
        h, w, _ = bgr.shape
        np.ascontiguousarray(bgr).tofile(self.d / "in.u8")
        self._run("yuv", self.d / "in.u8", w, h, self.d / "out.f32")
        return np.fromfile(self.d / "out.f32", np.float32).reshape(3, h, w)

    def resize(self, planes, dw, dh, interp):
        _, h, w = planes.shape
        np.ascontiguousarray(planes, np.float32).tofile(self.d / "in.f32")
        self._run("resize", self.d / "in.f32", w, h, dw, dh, interp, self.d / "out.f32")
        return np.fromfile(self.d / "out.f32", np.float32).reshape(3, dh, dw)

    def rgb8(self, planes):
        _, h, w = planes.shape
        np.ascontiguousarray(planes, np.float32).tofile(self.d / "in.f32")
        self._run("rgb8", self.d / "in.f32", w, h, self.d / "out.u8")
        return np.fromfile(self.d / "out.u8", np.uint8).reshape(h, w, 3)


def bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def check_stages(w2x, ctx, models, host, w, h, seed):
    """create -> denoise -> scale2x -> resize_linear -> download, each compared with the host path after every call."""
    bgr = np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
    img = w2x.Image(ctx, bgr)
    ref = host.yuv(bgr)
    assert bits_equal(img.planes(), ref), "create"
    img.denoise(models["noise1"])
    ref[0] = ctx.convert_plane(models["noise1"], ref[0])
    assert bits_equal(img.planes(), ref), "denoise"
    img.scale2x(models["scale2.0x"])
    y = ctx.convert_plane(models["scale2.0x"], host.resize(ref, 2 * w, 2 * h, "nearest")[0])
    ref = host.resize(ref, 2 * w, 2 * h, "cubic")
    ref[0] = y
    assert img.size() == (2 * w, 2 * h)
    assert bits_equal(img.planes(), ref), "scale2x"
    lw, lh = max(1, int(2 * w * 0.75)), max(1, int(2 * h * 0.75))
    img.resize_linear(lw, lh)
    ref = host.resize(ref, lw, lh, "linear")
    assert bits_equal(img.planes(), ref), "resize_linear"
    assert np.array_equal(img.download(), host.rgb8(ref)), "download"
    img.close()


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", SIZES, ids=[f"{w}x{h}" for w, h in SIZES])
def test_image_stages_bitwise_equal_host_path(w2x, models, driver, tmp_path, w, h):
    ctx = w2x.Context(0)
    check_stages(w2x, ctx, models, Host(driver, tmp_path), w, h, seed=w * 7 + h)
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["fp32_engine", "f16x3"])
def test_image_stages_other_engines(w2x, models, driver, tmp_path, variant):
    ctx = w2x.Context(0)
    if variant == "fp32_engine":
        ctx.set_engine(w2x.ENGINE_FP32)
    else:
        ctx.set_precision(w2x.PRECISION_F16X3)
    check_stages(w2x, ctx, models, Host(driver, tmp_path), 45, 33, seed=5)
    ctx.close()


@pytest.mark.gpu
def test_image_device_variants_on_a_caller_stream(w2x, models):
    torch = pytest.importorskip("torch")
    ctx = w2x.Context(0)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    w, h = 333, 217
    bgr = np.random.default_rng(9).integers(0, 256, (h, w, 3), dtype=np.uint8)
    padded = torch.zeros((h, w + 5, 3), dtype=torch.uint8, device="cuda")   # strided rows
    padded[:, :w] = torch.from_numpy(bgr).cuda()
    torch.cuda.synchronize()
    a = w2x.Image(ctx, bgr)
    b = w2x.Image.from_device(ctx, padded.data_ptr(), w, h, padded.stride(0))
    for img in (a, b):
        img.scale2x(models["scale2.0x"])
        img.resize_linear(500, 300)
    pa, pb = a.planes(), b.planes()
    assert bits_equal(pa, pb)
    out = torch.full((300, 500 + 3, 3), 7, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()                                                  # the fill ran on torch's stream, not the context's
    b.download_device(out.data_ptr(), out.stride(0))
    ctx.synchronize()
    assert np.array_equal(out[:, :500].cpu().numpy(), a.download())
    assert (out[:, 500:] == 7).all()                                          # the row padding is not written
    a.close()
    b.close()
    ctx.close()


@pytest.mark.gpu
def test_image_bad_arguments_and_context_lifetime(w2x, models):
    L = w2x.lib()
    import ctypes as C
    ctx = w2x.Context(0)
    px = np.zeros((4, 5, 3), np.uint8)
    out = C.c_void_p()
    p = C.c_void_p(px.ctypes.data)
    assert L.w2x_image_create(ctx._h, None, 5, 4, 15, C.byref(out)) == 1
    assert L.w2x_image_create(ctx._h, p, 0, 4, 15, C.byref(out)) == 1
    assert L.w2x_image_create(ctx._h, p, 5, -1, 15, C.byref(out)) == 1
    assert L.w2x_image_create(ctx._h, p, 5, 4, 14, C.byref(out)) == 1 and "stride" in L.w2x_last_error().decode()
    assert L.w2x_image_create_device(ctx._h, None, 5, 4, 15, C.byref(out)) == 1
    img = w2x.Image(ctx, px)
    for call in (lambda: img.resize_linear(0, 4), lambda: img.resize_linear(4, -2)):
        with pytest.raises(w2x.W2xError) as ei:
            call()
        assert ei.value.status == 1
    assert L.w2x_image_denoise(img._h, None) == 1
    assert L.w2x_image_download(img._h, None, 15) == 1
    assert L.w2x_image_download(img._h, p, 14) == 1
    assert L.w2x_image_planes(img._h, p, None, p, 20) == 1
    assert L.w2x_image_planes(img._h, p, p, p, 19) == 1
    rng = np.random.default_rng(0)
    two_in = w2x.Model.from_arrays([rng.normal(0, .1, (8, 2, 3, 3)), rng.normal(0, .1, (1, 8, 3, 3))], [np.zeros(8), np.zeros(1)])
    with pytest.raises(w2x.W2xError) as ei:
        img.scale2x(two_in)
    assert ei.value.status == 1 and "1 plane to 1 plane" in ei.value.message
    assert img.size() == (5, 4)                                               # a failed call leaves the image as it was
    # a context destroyed under a live image releases its memory; the image then refuses every call
    ctx.close()
    with pytest.raises(w2x.W2xError) as ei:
        img.size()
    assert ei.value.status == 1 and "context has been destroyed" in ei.value.message
    img.close()


@pytest.mark.gpu
def test_image_create_destroy_returns_device_memory(w2x):
    torch = pytest.importorskip("torch")
    ctx = w2x.Context(0)
    bgr = np.random.default_rng(1).integers(0, 256, (1080, 1920, 3), dtype=np.uint8)
    w2x.Image(ctx, bgr).close()                                               # module load, first allocations
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    for _ in range(20):
        w2x.Image(ctx, bgr).close()
    free1, _ = torch.cuda.mem_get_info()
    # 20 leaked 1080p images would be ~600 MB; other work on a shared GPU may move the figure by a little
    assert free0 - free1 < (32 << 20), (free0, free1)
    ctx.close()


# ---- the CLI: device path vs W2X_CLI_HOST_PLUMBING=1 ------------------------------------------------------------------
@pytest.fixture(scope="module")
def cli_env(w2x, json_models, tmp_path_factory):
    w2x.build()
    assert os.path.exists(CLI)
    d = tmp_path_factory.mktemp("cli_inputs")
    small = np.random.default_rng(11).integers(0, 256, (33, 45, 3), dtype=np.uint8)
    big = np.random.default_rng(4).integers(0, 256, (1080, 1920, 3), dtype=np.uint8)   # bench.py's config-2 image
    for name, a in (("small.ppm", small), ("big.ppm", big)):
        with open(d / name, "wb") as f:
            f.write(b"P6\n%d %d\n255\n" % (a.shape[1], a.shape[0]) + a.tobytes())
    return d, os.path.dirname(json_models["scale2.0x"])


def run_both(cli_env, tmp_path, image, mode, level, ratio):
    src, mdir = cli_env
    res = {}
    for path in ("device", "host"):
        d = tmp_path / path
        d.mkdir()
        os.symlink(src / image, d / image)
        env = dict(os.environ)
        env.pop("W2X_CLI_HOST_PLUMBING", None)
        if path == "host":
            env["W2X_CLI_HOST_PLUMBING"] = "1"
        r = subprocess.run([CLI, "-i", image, "-m", mode, "--noise_level", str(level), "--scale_ratio", str(ratio), "--model_dir", mdir],
                           capture_output=True, text=True, cwd=d, env=env, timeout=600)
        outs = sorted(f for f in os.listdir(d) if f != image)
        res[path] = (r.returncode, r.stdout.splitlines(), outs, {f: (d / f).read_bytes() for f in outs})
    dev, host = res["device"], res["host"]
    assert dev[0] == host[0] == 0, (dev[0], host[0])
    assert dev[1] == host[1]                                                  # stdout line for line
    assert dev[2] == host[2] and len(dev[2]) == 1                             # output names
    assert dev[3] == host[3]                                                  # the PNG files byte for byte (same pixels, same encoder)


CLI_SMALL = [(m, lv, r) for m in ("noise", "scale", "noise_scale") for lv in (1, 2) for r in (2.0, 3.0, 4.0, 1.5, 1.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode,level,ratio", CLI_SMALL)
def test_cli_device_path_equals_host_path_45x33(cli_env, tmp_path, mode, level, ratio):
    run_both(cli_env, tmp_path, "small.ppm", mode, level, ratio)


CLI_BIG = [("noise", 1, 2.0)] + [(m, 1, r) for m in ("scale", "noise_scale") for r in (2.0, 3.0, 4.0, 1.5, 1.0)]


@pytest.mark.gpu
@pytest.mark.slow
@pytest.mark.parametrize("mode,level,ratio", CLI_BIG)
def test_cli_device_path_equals_host_path_1920x1080(cli_env, tmp_path, mode, level, ratio):
    run_both(cli_env, tmp_path, "big.ppm", mode, level, ratio)
