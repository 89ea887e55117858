"""capi.py -- ctypes binding of include/w2x_b200.h (the reference-facing plugin surface).

Model        <-> std::vector<std::unique_ptr<w2xc::Model>> + modelUtility::generateModelFromJSON
Context.convert_plane  <-> w2xc::convertWithModels   (reference src/convertRoutine.hpp:25-28)
Context.filter_layer   <-> w2xc::Model::filter       (reference src/modelHandler.hpp:87-88)
set_jobs / set_block_size / ...  <-> w2xc::modelUtility setters (src/modelHandler.hpp:106-111)
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libw2x_b200.so")

ENGINE_AUTO, ENGINE_FP32, ENGINE_TC = 0, 1, 2
PRECISION_F16X3, PRECISION_F16_F8X2 = 0, 1
WALK_FUSED, WALK_BLOCKS = 0, 1

STATUS = {0: "W2X_OK", 1: "W2X_ERR_ARG", 2: "W2X_ERR_IO", 3: "W2X_ERR_PARSE", 4: "W2X_ERR_MODEL",
          5: "W2X_ERR_CUDA", 6: "W2X_ERR_NO_DEVICE", 7: "W2X_ERR_UNSUPPORTED", 8: "W2X_ERR_NOMEM"}

# every symbol include/w2x_b200.h declares (tests check the library exports all of them)
ABI_SYMBOLS = (
    "w2x_last_error", "w2x_version", "w2x_model_load_json", "w2x_model_create", "w2x_model_free",
    "w2x_model_layer_count", "w2x_model_layer_dims", "w2x_model_layer_params", "w2x_set_jobs", "w2x_get_jobs",
    "w2x_set_block_size", "w2x_set_block_size_exp2_square", "w2x_get_block_size", "w2x_requires_splitting",
    "w2x_block_table", "w2x_ctx_create", "w2x_ctx_destroy", "w2x_ctx_set_engine", "w2x_ctx_get_engine",
    "w2x_ctx_set_precision", "w2x_ctx_get_precision",
    "w2x_ctx_set_stream", "w2x_ctx_synchronize", "w2x_ctx_set_log", "w2x_ctx_set_block_walk",
    "w2x_ctx_set_scratch_limit", "w2x_convert_plane", "w2x_convert_plane_device", "w2x_filter_layer",
    "w2x_filter_layer_device", "w2x_convert_band_device", "w2x_ctx_launch_count", "w2x_ctx_set_timing",
    "w2x_ctx_layer_times", "w2x_ctx_layer_kernel_name", "w2x_band_create", "w2x_band_destroy", "w2x_band_load",
    "w2x_band_step", "w2x_band_halo", "w2x_band_finish", "w2x_band_load_rows", "w2x_band_export", "w2x_band_connect",
    "w2x_band_connect_local", "w2x_band_exchange", "w2x_band_run", "w2x_convert_tiles", "w2x_convert_tiles_async",
    "w2x_convert_tiles_device", "w2x_multi_create", "w2x_multi_destroy", "w2x_multi_device_count", "w2x_multi_ctx",
    "w2x_multi_set_precision", "w2x_multi_set_log", "w2x_multi_convert_plane", "w2x_multi_convert_tiles",
    "w2x_host_alloc", "w2x_host_free", "w2x_ctx_forget_model", "w2x_slab_create", "w2x_slab_destroy", "w2x_slab_export",
    "w2x_slab_connect", "w2x_slab_connect_local", "w2x_slab_convert", "w2x_slab_convert_async", "w2x_slab_synchronize",
    "w2x_image_create", "w2x_image_create_device", "w2x_image_destroy", "w2x_image_size", "w2x_image_denoise",
    "w2x_image_scale2x", "w2x_image_resize_linear", "w2x_image_download", "w2x_image_download_device", "w2x_image_planes",
)
BAND_BLOB_BYTES = 320


class W2xError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"{STATUS.get(status, status)}: {message}")
        self.status = status
        self.message = message


_lib = None
LOG_FN = C.CFUNCTYPE(None, C.c_char_p, C.c_void_p)


def lib_path() -> str:
    return _LIB_PATH


def lib():
    """Load libw2x_b200.so.  Fails loudly when it has not been built: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise W2xError(-1, f"{_LIB_PATH} is missing -- run `python waifu2x-converter-cpp_b200/build.py` "
                           "(the product has no Python/CPU fallback)")
    L = C.CDLL(_LIB_PATH)
    vp, ci, cs, fp = C.c_void_p, C.c_int, C.c_size_t, C.POINTER(C.c_float)
    L.w2x_last_error.restype = C.c_char_p
    L.w2x_version.restype = C.c_char_p
    L.w2x_model_load_json.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.w2x_model_create.argtypes = [ci, C.POINTER(ci), C.POINTER(ci), C.POINTER(fp), C.POINTER(C.POINTER(C.c_double)),
                                   C.POINTER(vp)]
    L.w2x_model_free.argtypes = [vp]
    L.w2x_model_free.restype = None
    L.w2x_model_layer_count.argtypes = [vp]
    L.w2x_model_layer_dims.argtypes = [vp, ci, C.POINTER(ci), C.POINTER(ci), C.POINTER(ci)]
    L.w2x_model_layer_params.argtypes = [vp, ci, C.POINTER(fp), C.POINTER(C.POINTER(C.c_double))]
    L.w2x_set_jobs.argtypes = [ci]
    L.w2x_set_block_size.argtypes = [ci, ci]
    L.w2x_set_block_size_exp2_square.argtypes = [ci]
    L.w2x_get_block_size.argtypes = [C.POINTER(ci), C.POINTER(ci)]
    L.w2x_get_block_size.restype = None
    L.w2x_requires_splitting.argtypes = [ci, ci]
    L.w2x_block_table.argtypes = [ci, ci, ci, C.POINTER(ci), ci, C.POINTER(ci), C.POINTER(ci)]
    L.w2x_ctx_create.argtypes = [ci, C.POINTER(vp)]
    L.w2x_ctx_destroy.argtypes = [vp]
    L.w2x_ctx_destroy.restype = None
    L.w2x_ctx_set_engine.argtypes = [vp, ci]
    L.w2x_ctx_get_engine.argtypes = [vp]
    L.w2x_ctx_set_precision.argtypes = [vp, ci]
    L.w2x_ctx_get_precision.argtypes = [vp]
    L.w2x_ctx_set_stream.argtypes = [vp, vp]
    L.w2x_ctx_synchronize.argtypes = [vp]
    L.w2x_ctx_set_log.argtypes = [vp, LOG_FN, vp]
    L.w2x_ctx_set_block_walk.argtypes = [vp, ci]
    L.w2x_ctx_set_scratch_limit.argtypes = [vp, cs]
    L.w2x_convert_plane.argtypes = [vp, vp, vp, ci, ci, cs, vp, cs, ci]
    L.w2x_convert_plane_device.argtypes = [vp, vp, vp, ci, ci, cs, vp, cs, ci]
    L.w2x_convert_band_device.argtypes = [vp, vp, vp, ci, ci, ci, ci, cs, vp, cs]
    L.w2x_filter_layer.argtypes = [vp, vp, ci, C.POINTER(vp), ci, C.POINTER(vp), ci, ci, ci, cs, cs]
    L.w2x_filter_layer_device.argtypes = [vp, vp, ci, vp, vp, ci, ci]
    L.w2x_ctx_launch_count.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.w2x_ctx_set_timing.argtypes = [vp, ci]
    L.w2x_ctx_layer_times.argtypes = [vp, ci, fp, C.POINTER(ci), C.POINTER(ci), ci]
    L.w2x_ctx_layer_kernel_name.argtypes = [vp, ci]
    L.w2x_ctx_layer_kernel_name.restype = C.c_char_p
    L.w2x_band_create.argtypes = [vp, vp, ci, ci, ci, ci, C.POINTER(vp)]
    L.w2x_band_destroy.argtypes = [vp]
    L.w2x_band_destroy.restype = None
    L.w2x_band_load.argtypes = [vp, vp, cs]
    L.w2x_band_step.argtypes = [vp, ci]
    L.w2x_band_halo.argtypes = [vp, ci, C.POINTER(ci), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(cs)]
    L.w2x_band_finish.argtypes = [vp, vp, cs]
    L.w2x_ctx_forget_model.argtypes = [vp, vp]
    L.w2x_slab_create.argtypes = [vp, vp, ci, ci, ci, ci, ci, ci, C.POINTER(vp)]
    L.w2x_slab_destroy.argtypes = [vp]
    L.w2x_slab_destroy.restype = None
    L.w2x_slab_export.argtypes = [vp, vp]
    L.w2x_slab_connect.argtypes = [vp, vp, vp]
    L.w2x_slab_connect_local.argtypes = [vp, vp, vp]
    L.w2x_slab_convert.argtypes = [vp, vp, cs, vp, cs]
    L.w2x_slab_convert_async.argtypes = [vp, vp, cs, vp, cs]
    L.w2x_slab_synchronize.argtypes = [vp]
    L.w2x_host_alloc.argtypes = [cs]
    L.w2x_host_alloc.restype = vp
    L.w2x_host_free.argtypes = [vp]
    L.w2x_host_free.restype = None
    L.w2x_band_load_rows.argtypes = [vp, vp, cs]
    L.w2x_band_export.argtypes = [vp, vp]
    L.w2x_band_connect.argtypes = [vp, vp, vp]
    L.w2x_band_connect_local.argtypes = [vp, vp, vp]
    L.w2x_band_exchange.argtypes = [vp, ci]
    L.w2x_band_run.argtypes = [vp, vp, cs, vp, cs]
    L.w2x_convert_tiles.argtypes = [vp, vp, C.POINTER(vp), C.POINTER(vp), ci, ci, ci, cs, cs]
    L.w2x_convert_tiles_async.argtypes = [vp, vp, C.POINTER(vp), C.POINTER(vp), ci, ci, ci, cs, cs]
    L.w2x_convert_tiles_device.argtypes = [vp, vp, vp, vp, ci, ci, ci]
    L.w2x_multi_create.argtypes = [C.POINTER(ci), ci, C.POINTER(vp)]
    L.w2x_multi_destroy.argtypes = [vp]
    L.w2x_multi_destroy.restype = None
    L.w2x_multi_device_count.argtypes = [vp]
    L.w2x_multi_ctx.argtypes = [vp, ci]
    L.w2x_multi_ctx.restype = vp
    L.w2x_multi_set_precision.argtypes = [vp, ci]
    L.w2x_multi_set_log.argtypes = [vp, LOG_FN, vp]
    L.w2x_multi_convert_plane.argtypes = [vp, vp, vp, ci, ci, cs, vp, cs, ci]
    L.w2x_multi_convert_tiles.argtypes = [vp, vp, C.POINTER(vp), C.POINTER(vp), ci, ci, ci, cs, cs]
    L.w2x_image_create.argtypes = [vp, vp, ci, ci, cs, C.POINTER(vp)]
    L.w2x_image_create_device.argtypes = [vp, vp, ci, ci, cs, C.POINTER(vp)]
    L.w2x_image_destroy.argtypes = [vp]
    L.w2x_image_destroy.restype = None
    L.w2x_image_size.argtypes = [vp, C.POINTER(ci), C.POINTER(ci)]
    L.w2x_image_denoise.argtypes = [vp, vp]
    L.w2x_image_scale2x.argtypes = [vp, vp]
    L.w2x_image_resize_linear.argtypes = [vp, ci, ci]
    L.w2x_image_download.argtypes = [vp, vp, cs]
    L.w2x_image_download_device.argtypes = [vp, vp, cs]
    L.w2x_image_planes.argtypes = [vp, vp, vp, vp, cs]
    L.w2x_debug_set_host_bands.argtypes = [vp, ci]
    L.w2x_debug_set_pair.argtypes = [vp, ci]
    L.w2x_debug_set_fuse_last.argtypes = [vp, ci]
    L.w2x_debug_set_num_sms.argtypes = [vp, ci]
    L.w2x_debug_tc_pack8.argtypes = [vp, ci, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(cs)]
    L.w2x_debug_tc_strip.argtypes = [vp, ci, ci, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(cs)]
    L.w2x_debug_set_strip.argtypes = [vp, ci]
    L.w2x_debug_tc_profile_enable.argtypes = [vp, ci]
    L.w2x_debug_tc_profile_read.argtypes = [vp, ci, C.POINTER(C.c_uint64), C.POINTER(ci)]
    L.w2x_debug_tc_pack.argtypes = [vp, ci, C.POINTER(C.POINTER(C.c_uint16)), C.POINTER(cs), C.POINTER(ci), C.POINTER(ci),
                                    C.POINTER(C.c_float), C.POINTER(ci)]
    _lib = L
    return L


def _check(status):
    if status != 0:
        raise W2xError(status, lib().w2x_last_error().decode("utf-8", "replace"))


def version() -> str:
    return lib().w2x_version().decode()


# ---- modelUtility ------------------------------------------------------------------------------
def set_jobs(n): _check(lib().w2x_set_jobs(n))
def get_jobs(): return lib().w2x_get_jobs()
def set_block_size(w, h): _check(lib().w2x_set_block_size(w, h))
def set_block_size_exp2_square(e): _check(lib().w2x_set_block_size_exp2_square(e))


def get_block_size():
    w, h = C.c_int(), C.c_int()
    lib().w2x_get_block_size(C.byref(w), C.byref(h))
    return w.value, h.value


def requires_splitting(w, h) -> bool:
    return bool(lib().w2x_requires_splitting(w, h))


def block_table(w, h, n_model=7):
    """-> (int32 array [n_blocks, 8], split_cols, split_rows); rows are
    (r, c, in_y0, in_y1, in_x0, in_x1, out_y0, out_x0) in the reference's processing order."""
    sc, sr = C.c_int(), C.c_int()
    n = lib().w2x_block_table(w, h, n_model, None, 0, C.byref(sc), C.byref(sr))
    if n < 0:
        raise W2xError(-n, lib().w2x_last_error().decode())
    tab = np.zeros((n, 8), np.int32)
    lib().w2x_block_table(w, h, n_model, tab.ctypes.data_as(C.POINTER(C.c_int)), n, None, None)
    return tab, sc.value, sr.value


# ---- Model --------------------------------------------------------------------------------------
class Model:
    def __init__(self, handle):
        self._h = handle

    @classmethod
    def load_json(cls, path):
        h = C.c_void_p()
        _check(lib().w2x_model_load_json(os.fsencode(path), C.byref(h)))
        return cls(h)

    @classmethod
    def from_arrays(cls, weights, biases):
        n = len(weights)
        ws = [np.ascontiguousarray(w, np.float32) for w in weights]
        bs = [np.ascontiguousarray(b, np.float64) for b in biases]
        n_in = (C.c_int * n)(*[w.shape[1] for w in ws])
        n_out = (C.c_int * n)(*[w.shape[0] for w in ws])
        wp = (C.POINTER(C.c_float) * n)(*[w.ctypes.data_as(C.POINTER(C.c_float)) for w in ws])
        bp = (C.POINTER(C.c_double) * n)(*[b.ctypes.data_as(C.POINTER(C.c_double)) for b in bs])
        h = C.c_void_p()
        _check(lib().w2x_model_create(n, n_in, n_out, wp, bp, C.byref(h)))
        return cls(h)

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.w2x_model_free(self._h)
            self._h = None

    def __len__(self):
        return lib().w2x_model_layer_count(self._h)

    def dims(self, layer):
        a, b, k = C.c_int(), C.c_int(), C.c_int()
        _check(lib().w2x_model_layer_dims(self._h, layer, C.byref(a), C.byref(b), C.byref(k)))
        return a.value, b.value, k.value

    def params(self, layer):
        n_in, n_out, k = self.dims(layer)
        wp, bp = C.POINTER(C.c_float)(), C.POINTER(C.c_double)()
        _check(lib().w2x_model_layer_params(self._h, layer, C.byref(wp), C.byref(bp)))
        w = np.ctypeslib.as_array(wp, shape=(n_out, n_in, k, k)).copy()
        b = np.ctypeslib.as_array(bp, shape=(n_out,)).copy()
        return w, b


    def debug_tc_pack(self, layer):
        """(fp16 bit patterns [chunk][tap][kblock][hi|lo][n_out*32], n_chunk, kblocks, wscale) -- packing tests only."""
        dp, n = C.POINTER(C.c_uint16)(), C.c_size_t()
        kc, nch, ws, kbl = C.c_int(), C.c_int(), C.c_float(), C.c_int()
        _check(lib().w2x_debug_tc_pack(self._h, layer, C.byref(dp), C.byref(n), C.byref(kc), C.byref(nch), C.byref(ws), C.byref(kbl)))
        if n.value == 0:
            return None, nch.value, kbl.value, ws.value
        assert kc.value == 32
        return np.ctypeslib.as_array(dp, shape=(n.value,)).copy(), nch.value, kbl.value, ws.value


    def debug_tc_pack8(self, layer):
        """uint8 image [chunk][tap][kblock][wh fp16 n_out*64 B | wh8 n_out*32 B | wl8 n_out*32 B] of the f8 flavour."""
        dp, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        _check(lib().w2x_debug_tc_pack8(self._h, layer, C.byref(dp), C.byref(n)))
        return None if n.value == 0 else np.ctypeslib.as_array(dp, shape=(n.value,)).copy()


    def debug_tc_strip(self, layer, f8):
        """uint8 image of the row-strip kernel's weights: [chunk][kx] stages, rows ky-major; None for the wide layers."""
        dp, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        _check(lib().w2x_debug_tc_strip(self._h, layer, int(f8), C.byref(dp), C.byref(n)))
        return None if n.value == 0 else np.ctypeslib.as_array(dp, shape=(n.value,)).copy()


# ---- Context ------------------------------------------------------------------------------------
class Context:
    def __init__(self, device=0, engine=ENGINE_AUTO):
        h = C.c_void_p()
        _check(lib().w2x_ctx_create(device, C.byref(h)))
        self._h = h
        self._log_cb = None
        if engine != ENGINE_AUTO:
            self.set_engine(engine)

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.w2x_ctx_destroy(self._h)
            self._h = None

    __del__ = close

    def set_engine(self, engine): _check(lib().w2x_ctx_set_engine(self._h, engine))
    def forget_model(self, model): _check(lib().w2x_ctx_forget_model(self._h, model._h))
    def set_precision(self, precision): _check(lib().w2x_ctx_set_precision(self._h, precision))
    def get_precision(self): return lib().w2x_ctx_get_precision(self._h)
    def set_stream(self, stream_ptr): _check(lib().w2x_ctx_set_stream(self._h, C.c_void_p(stream_ptr)))
    def synchronize(self): _check(lib().w2x_ctx_synchronize(self._h))
    def set_block_walk(self, mode): _check(lib().w2x_ctx_set_block_walk(self._h, mode))
    def set_scratch_limit(self, nbytes): _check(lib().w2x_ctx_set_scratch_limit(self._h, nbytes))
    def set_timing(self, on): _check(lib().w2x_ctx_set_timing(self._h, int(on)))

    def debug_set_pair(self, on): _check(lib().w2x_debug_set_pair(self._h, int(on)))
    def debug_set_strip(self, on): _check(lib().w2x_debug_set_strip(self._h, int(on)))
    def debug_set_host_bands(self, n): _check(lib().w2x_debug_set_host_bands(self._h, n))
    def debug_set_fuse_last(self, on): _check(lib().w2x_debug_set_fuse_last(self._h, int(on)))
    def debug_set_num_sms(self, n): _check(lib().w2x_debug_set_num_sms(self._h, int(n)))
    def debug_tc_profile_enable(self, on=True): _check(lib().w2x_debug_tc_profile_enable(self._h, int(on)))

    def debug_tc_profile_read(self, layer):
        """per-role cycle counters of the tcgen05 kernel of `layer`, averaged per CTA (dict)."""
        out = (C.c_uint64 * 16)()
        n = C.c_int()
        _check(lib().w2x_debug_tc_profile_read(self._h, layer, out, C.byref(n)))
        names = ["total", "mma_wait_acc", "mma_wait_a", "mma_wait_b", "aprod_wait", "bprod_wait", "epi_wait", "epi_work", "tilesets"]
        d = {k: out[i] / max(n.value, 1) for i, k in enumerate(names)}
        d["ctas"] = n.value
        return d

    def set_log(self, fn):
        """fn(str) receives the reference's progress lines; None disables."""
        if fn is None:
            self._log_cb = LOG_FN()
        else:
            self._log_cb = LOG_FN(lambda line, _u: fn(line.decode()))
        _check(lib().w2x_ctx_set_log(self._h, self._log_cb, None))

    def launch_count(self):
        n = C.c_uint64()
        _check(lib().w2x_ctx_launch_count(self._h, C.byref(n)))
        return n.value

    def layer_times(self, reset=True, max_layers=16):
        ms = (C.c_float * max_layers)()
        cnt = (C.c_int * max_layers)()
        n = C.c_int()
        _check(lib().w2x_ctx_layer_times(self._h, max_layers, ms, cnt, C.byref(n), int(reset)))
        return [(ms[i], cnt[i], lib().w2x_ctx_layer_kernel_name(self._h, i).decode()) for i in range(n.value)]

    # w2xc::convertWithModels on a host numpy plane (copies are inside the call)
    def convert_plane(self, model: Model, plane, block_splitting=True, out=None):
        x = np.asarray(plane, np.float32)
        if x.ndim != 2:
            raise ValueError("plane must be 2-D")
        if x.strides[1] != 4 or x.strides[0] % 4 or x.strides[0] < x.shape[1] * 4:
            x = np.ascontiguousarray(x)
        h, w = x.shape
        if out is None:
            out = np.empty((h, w), np.float32)
        _check(lib().w2x_convert_plane(self._h, model._h, C.c_void_p(x.ctypes.data), w, h, x.strides[0],
                                       C.c_void_p(out.ctypes.data), out.strides[0], int(bool(block_splitting))))
        return out

    # device pointers (ints), asynchronous on the context's stream
    def convert_plane_device(self, model: Model, d_in, w, h, in_stride_bytes, d_out, out_stride_bytes,
                             block_splitting=True):
        _check(lib().w2x_convert_plane_device(self._h, model._h, C.c_void_p(d_in), w, h, in_stride_bytes,
                                              C.c_void_p(d_out), out_stride_bytes, int(bool(block_splitting))))

    def convert_band_device(self, model: Model, d_in, w, band_h, rows_above, rows_below, in_stride_bytes, d_out,
                            out_stride_bytes):
        _check(lib().w2x_convert_band_device(self._h, model._h, C.c_void_p(d_in), w, band_h, rows_above, rows_below,
                                             in_stride_bytes, C.c_void_p(d_out), out_stride_bytes))

    # n independent planes of one shape in one batched pass (the reference's block loop; BASELINE config 5)
    def convert_tiles(self, model: Model, tiles, out=None):
        x = np.ascontiguousarray(tiles, np.float32)
        if x.ndim != 3:
            raise ValueError("tiles must be [n][h][w]")
        n, h, w = x.shape
        if out is None:
            out = np.empty_like(x)
        ip = (C.c_void_p * n)(*[x[i].ctypes.data for i in range(n)])
        op = (C.c_void_p * n)(*[out[i].ctypes.data for i in range(n)])
        _check(lib().w2x_convert_tiles(self._h, model._h, ip, op, n, w, h, w * 4, w * 4))
        return out

    def convert_tiles_device(self, model: Model, d_in, d_out, n, w, h):
        _check(lib().w2x_convert_tiles_device(self._h, model._h, C.c_void_p(d_in), C.c_void_p(d_out), n, w, h))

    # w2xc::Model::filter on host planes [n_in][h][w] -> [n_out][h][w]
    def filter_layer(self, model: Model, layer, in_planes):
        x = np.ascontiguousarray(in_planes, np.float32)
        n_in, n_out, _ = model.dims(layer)
        _, h, w = x.shape
        out = np.empty((n_out, h, w), np.float32)
        ip = (C.c_void_p * x.shape[0])(*[x[i].ctypes.data for i in range(x.shape[0])])
        op = (C.c_void_p * n_out)(*[out[i].ctypes.data for i in range(n_out)])
        _check(lib().w2x_filter_layer(self._h, model._h, layer, ip, x.shape[0], op, n_out, w, h, w * 4, w * 4))
        return out

    def filter_layer_device(self, model: Model, layer, d_in, d_out, w, h):
        _check(lib().w2x_filter_layer_device(self._h, model._h, layer, C.c_void_p(d_in), C.c_void_p(d_out), w, h))


# ---- whole images on the device -----------------------------------------------------------------
class Image:
    """w2x_image_*: an 8-bit B,G,R image kept on the context's device as fp32 Y, U, V planes through the reference
    main.cpp's phases (denoise, 2x scaling, bilinear shrink), bit-identical to the host plumbing.

    Image(ctx, bgr)                          from a host uint8 array [h][w][3] (rows may be strided)
    Image.from_device(ctx, ptr, w, h, stride)  from device pixels (e.g. a CUDA uint8 tensor's data_ptr()), asynchronous"""

    def __init__(self, ctx: Context, bgr=None, _handle=None):
        self._ctx = ctx                      # the context must outlive the image
        if _handle is not None:
            self._h = _handle
            return
        x = np.asarray(bgr, np.uint8)
        if x.ndim != 3 or x.shape[2] != 3:
            raise ValueError("bgr must be [h][w][3] uint8")
        if x.strides[2] != 1 or x.strides[1] != 3:
            x = np.ascontiguousarray(x)
        h = C.c_void_p()
        _check(lib().w2x_image_create(ctx._h, C.c_void_p(x.ctypes.data), x.shape[1], x.shape[0], x.strides[0], C.byref(h)))
        self._h = h

    @classmethod
    def from_device(cls, ctx: Context, d_bgr, width, height, stride_bytes):
        h = C.c_void_p()
        _check(lib().w2x_image_create_device(ctx._h, C.c_void_p(d_bgr), width, height, stride_bytes, C.byref(h)))
        return cls(ctx, _handle=h)

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.w2x_image_destroy(self._h)
            self._h = None

    __del__ = close

    def size(self):
        """-> (width, height)"""
        w, h = C.c_int(), C.c_int()
        _check(lib().w2x_image_size(self._h, C.byref(w), C.byref(h)))
        return w.value, h.value

    def denoise(self, model: Model): _check(lib().w2x_image_denoise(self._h, model._h))
    def scale2x(self, model: Model): _check(lib().w2x_image_scale2x(self._h, model._h))
    def resize_linear(self, width, height): _check(lib().w2x_image_resize_linear(self._h, width, height))

    def download(self, out=None):
        """-> uint8 [h][w][3] B,G,R (host, synchronous)"""
        w, h = self.size()
        if out is None:
            out = np.empty((h, w, 3), np.uint8)
        _check(lib().w2x_image_download(self._h, C.c_void_p(out.ctypes.data), out.strides[0]))
        return out

    def download_device(self, d_bgr, stride_bytes):
        _check(lib().w2x_image_download_device(self._h, C.c_void_p(d_bgr), stride_bytes))

    def planes(self):
        """-> float32 [3][h][w]: Y, U, V (host, synchronous)"""
        w, h = self.size()
        out = np.empty((3, h, w), np.float32)
        _check(lib().w2x_image_planes(self._h, C.c_void_p(out[0].ctypes.data), C.c_void_p(out[1].ctypes.data),
                                      C.c_void_p(out[2].ctypes.data), w * 4))
        return out


# ---- row-band session with a halo exchange between layers ---------------------------------------
class DevBytes:
    """Zero-copy view of a device range for torch.as_tensor (CUDA array interface, uint8)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


class Band:
    """w2x_band_*: one rank's rows of a plane, intermediate activations exchanged row-wise between layers."""

    def __init__(self, ctx: Context, model: Model, width, band_rows, has_up, has_down):
        h = C.c_void_p()
        _check(lib().w2x_band_create(ctx._h, model._h, width, band_rows, int(has_up), int(has_down), C.byref(h)))
        self._h, self._ctx, self._model = h, ctx, model
        self.steps = len(model) - 1          # w2x_band_step(0 .. n-2), then finish

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.w2x_band_destroy(self._h)
            self._h = None

    __del__ = close

    def load(self, d_in, in_stride_bytes): _check(lib().w2x_band_load(self._h, C.c_void_p(d_in), in_stride_bytes))
    def step(self, k): _check(lib().w2x_band_step(self._h, k))
    def finish(self, d_out, out_stride_bytes): _check(lib().w2x_band_finish(self._h, C.c_void_p(d_out), out_stride_bytes))

    def load_rows(self, d_in, in_stride_bytes): _check(lib().w2x_band_load_rows(self._h, C.c_void_p(d_in), in_stride_bytes))
    def exchange(self, k): _check(lib().w2x_band_exchange(self._h, k))

    def run(self, d_in, in_stride_bytes, d_out, out_stride_bytes):
        """One pass of a connected band: own rows in, own rows out (exchanges inside the library, peer memory)."""
        _check(lib().w2x_band_run(self._h, C.c_void_p(d_in), in_stride_bytes, C.c_void_p(d_out), out_stride_bytes))

    def export(self) -> bytes:
        buf = C.create_string_buffer(BAND_BLOB_BYTES)
        _check(lib().w2x_band_export(self._h, buf))
        return buf.raw

    def connect(self, up_blob, down_blob):
        """Map the neighbour ranks' sessions (CUDA IPC); blobs come from their export()."""
        _check(lib().w2x_band_connect(self._h, up_blob, down_blob))

    def connect_local(self, up, down):
        _check(lib().w2x_band_connect_local(self._h, up._h if up is not None else None, down._h if down is not None else None))

    def halo(self, k):
        """-> list of (send_up, recv_up, send_down, recv_down, nbytes) device-pointer tuples (None = no neighbour)."""
        n, nb = C.c_int(), C.c_size_t()
        su, ru, sd, rd = ((C.c_void_p * 4)() for _ in range(4))
        _check(lib().w2x_band_halo(self._h, k, C.byref(n), su, ru, sd, rd, C.byref(nb)))
        return [(su[i], ru[i], sd[i], rd[i], nb.value) for i in range(n.value)]


class Slab:
    """w2x_slab_*: one rank's rows of a multi-GPU plane with HOST buffers; upload / layers / download pipelined over sub-bands."""

    def __init__(self, ctx: Context, model: Model, width, rows, has_up, has_down, order=0, n_sub=0):
        h = C.c_void_p()
        _check(lib().w2x_slab_create(ctx._h, model._h, width, rows, int(has_up), int(has_down), int(order), int(n_sub), C.byref(h)))
        self._h, self._ctx, self._model = h, ctx, model

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.w2x_slab_destroy(self._h)
            self._h = None

    __del__ = close

    def export(self) -> bytes:
        buf = C.create_string_buffer(2 * BAND_BLOB_BYTES)
        _check(lib().w2x_slab_export(self._h, buf))
        return buf.raw

    def connect(self, up_blob, down_blob): _check(lib().w2x_slab_connect(self._h, up_blob, down_blob))

    def connect_local(self, up, down):
        _check(lib().w2x_slab_connect_local(self._h, up._h if up is not None else None, down._h if down is not None else None))

    def convert(self, rows_in, rows_out):
        """numpy [rows][width] fp32 (pinned for full overlap) -> rows_out"""
        _check(lib().w2x_slab_convert(self._h, C.c_void_p(rows_in.ctypes.data), rows_in.strides[0], C.c_void_p(rows_out.ctypes.data), rows_out.strides[0]))
        return rows_out

    def convert_async(self, rows_in, rows_out):
        _check(lib().w2x_slab_convert_async(self._h, C.c_void_p(rows_in.ctypes.data), rows_in.strides[0], C.c_void_p(rows_out.ctypes.data), rows_out.strides[0]))

    def synchronize(self): _check(lib().w2x_slab_synchronize(self._h))


# ---- one process, N GPUs ------------------------------------------------------------------------
class Multi:
    """w2x_multi_*: N contexts driven by one host thread (row bands + peer-memory halo exchange, or tile-per-GPU)."""

    def __init__(self, devices):
        devs = list(devices)
        arr = (C.c_int * len(devs))(*devs)
        h = C.c_void_p()
        _check(lib().w2x_multi_create(arr, len(devs), C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.w2x_multi_destroy(self._h)
            self._h = None

    __del__ = close

    def set_precision(self, precision): _check(lib().w2x_multi_set_precision(self._h, precision))

    def convert_plane(self, model: Model, plane, block_splitting=True, out=None):
        x = np.ascontiguousarray(plane, np.float32)
        h, w = x.shape
        if out is None:
            out = np.empty((h, w), np.float32)
        _check(lib().w2x_multi_convert_plane(self._h, model._h, C.c_void_p(x.ctypes.data), w, h, x.strides[0],
                                             C.c_void_p(out.ctypes.data), out.strides[0], int(bool(block_splitting))))
        return out

    def convert_tiles(self, model: Model, tiles, out=None):
        x = np.ascontiguousarray(tiles, np.float32)
        n, h, w = x.shape
        if out is None:
            out = np.empty_like(x)
        ip = (C.c_void_p * n)(*[x[i].ctypes.data for i in range(n)])
        op = (C.c_void_p * n)(*[out[i].ctypes.data for i in range(n)])
        _check(lib().w2x_multi_convert_tiles(self._h, model._h, ip, op, n, w, h, w * 4, w * 4))
        return out
