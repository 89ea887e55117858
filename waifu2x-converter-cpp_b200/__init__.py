"""waifu2x-converter-cpp_b200 -- the B200-native convolution hot path of waifu2x-converter-cpp.

The product is the C-ABI shared library built from csrc/ (declared in include/w2x_b200.h).  This
package is only the Python binding to it (ctypes, capi.py) plus the in-tree build recipe
(build.py).  Importing it never touches oracle/ and never falls back to CPU arithmetic: every
compute call goes to libw2x_b200.so, which fails with W2X_ERR_NO_DEVICE without an sm_100 GPU.

The directory name is not a valid Python identifier; load it with

    import importlib.util, sys
    spec = importlib.util.spec_from_file_location(
        "w2x_b200", "<repo>/waifu2x-converter-cpp_b200/__init__.py",
        submodule_search_locations=["<repo>/waifu2x-converter-cpp_b200"])
    w2x_b200 = importlib.util.module_from_spec(spec); sys.modules["w2x_b200"] = w2x_b200
    spec.loader.exec_module(w2x_b200)

(tests/conftest.py, bench.py and __graft_entry__.py do exactly this through w2x_loader.py).
"""
from .capi import (  # noqa: F401
    ENGINE_AUTO, ENGINE_FP32, ENGINE_TC, PRECISION_F16X3, PRECISION_F16_F8X2, WALK_BLOCKS, WALK_FUSED, Band, Context, DevBytes, Image, Model, Multi, Slab, W2xError,
    block_table, get_block_size, get_jobs, lib, lib_path, requires_splitting, set_block_size,
    set_block_size_exp2_square, set_jobs, version,
)
from .build import build  # noqa: F401
