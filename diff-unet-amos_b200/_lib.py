"""ctypes binding of libdunet_b200.so (C ABI: include/dunet.h).

There is NO fallback: if the CUDA library cannot be loaded the import of the compute entry points raises.  The only
PyTorch involvement is device memory (tensor.data_ptr()) and the current CUDA stream handle.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int32, c_int64, c_size_t, c_uint8, c_uint32, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdunet_b200.so")
DUNET_VERSION = 230  # include/dunet.h: the ABI the signatures below describe
MAX_IN_CHANNELS = 10  # include/dunet.h DUNET_MAX_IN_CHANNELS

DUNET_FLAG_REF_CONV = 1
DUNET_FLAG_KEEP_FP32_WEIGHTS = 2
DUNET_FLAG_GENERIC_CONV = 4
DUNET_FLAG_DUAL_STREAM = 8
DUNET_FLAG_FP32X3 = 16
DUNET_FLAG_NO_FUSED_NORM = 32
DUNET_FLAG_TC64_CB64 = 64
DUNET_FLAG_FP16 = 128
DUNET_FLAG_PLAIN_ENCODER = 256


class DunetCfg(ctypes.Structure):
    _fields_ = [
        ("num_classes", c_int32),
        ("in_channels", c_int32),
        ("patch", c_int32 * 3),
        ("features", c_int32 * 6),
        ("batch_max", c_int32),
        ("num_steps", c_int32),
        ("flags", c_uint32),
    ]


class DunetError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libdunet_b200 error {code}: {msg}")
        self.code = code


# every symbol include/dunet.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "dunet_version": (c_int32, []),
    "dunet_last_error": (c_char_p, []),
    "dunet_plan_create": (c_int32, [POINTER(c_void_p), POINTER(DunetCfg)]),
    "dunet_plan_destroy": (None, [c_void_p]),
    "dunet_plan_set_weight": (c_int32, [c_void_p, c_char_p, c_void_p, POINTER(c_int64), c_int32, c_void_p]),
    "dunet_plan_set_schedule": (c_int32, [c_void_p, c_int32, POINTER(c_int32), POINTER(c_float), POINTER(c_float), POINTER(c_float)]),
    "dunet_plan_commit": (c_int32, [c_void_p, c_void_p]),
    "dunet_workspace_bytes": (c_int32, [c_void_p, c_int32, POINTER(c_size_t)]),
    "dunet_encode": (c_int32, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p]),
    "dunet_get_embedding": (c_int32, [c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_void_p]),
    "dunet_set_embedding": (c_int32, [c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_void_p]),
    "dunet_denoise_step": (c_int32, [c_void_p, c_void_p, c_void_p, POINTER(c_int32), c_void_p, c_int32, c_void_p, c_void_p]),
    "dunet_ddim_sample": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_float, c_int32, c_void_p, c_void_p]),
    "dunet_crop_window": (c_int32, [c_void_p, POINTER(c_int32), c_void_p, POINTER(c_int32), POINTER(c_int32), c_void_p]),
    "dunet_zero": (c_int32, [c_void_p, c_size_t, c_void_p]),
    "dunet_crop_windows": (c_int32, [c_void_p, POINTER(c_int32), c_void_p, POINTER(c_int32), POINTER(c_int32), c_int32, c_void_p]),
    "dunet_infer_windows": (c_int32, [c_void_p, c_void_p, POINTER(c_int32), POINTER(c_int32), c_int32, c_void_p, c_uint64, POINTER(c_int64),
                                      c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dunet_stitch_add": (c_int32, [c_void_p, POINTER(c_int32), c_int32, c_void_p, POINTER(c_int32), POINTER(c_int32), c_void_p]),
    "dunet_finalize": (c_int32, [c_void_p, POINTER(c_int32), c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dunet_stitch_add_weighted": (c_int32, [c_void_p, c_void_p, POINTER(c_int32), c_int32, c_void_p, c_void_p, POINTER(c_int32), POINTER(c_int32), c_void_p]),
    "dunet_finalize_weighted": (c_int32, [c_void_p, c_void_p, POINTER(c_int32), c_int32, c_void_p, c_void_p, c_void_p]),
    "dunet_scale_intensity": (c_int32, [c_void_p, c_void_p, c_int64, c_float, c_float, c_float, c_float, c_int32, c_void_p]),
    "dunet_foreground_bbox": (c_int32, [c_void_p, c_int32, POINTER(c_int32), c_void_p, c_void_p]),
    "dunet_crop_box": (c_int32, [c_void_p, c_int32, POINTER(c_int32), c_void_p, POINTER(c_int32), POINTER(c_int32), c_void_p]),
    "dunet_resample_spacing": (c_int32, [c_void_p, c_int32, POINTER(c_int32), c_void_p, POINTER(c_int32), POINTER(ctypes.c_double), c_int32, c_void_p]),
    "dunet_invert_labels": (c_int32, [c_void_p, c_int32, POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), POINTER(ctypes.c_double),
                                      POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), c_int32, c_void_p, c_void_p, c_void_p]),
    "dunet_uncertainty_fuse": (c_int32, [c_void_p, c_int32, c_int32, c_int64, c_void_p, c_void_p]),
    "dunet_finalize_peers": (c_int32, [POINTER(c_void_p), POINTER(c_int32), POINTER(c_int32), c_int32, POINTER(c_int32), c_int32, c_int32,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dunet_ipc_alloc": (c_int32, [POINTER(c_void_p), c_size_t, POINTER(c_uint8)]),
    "dunet_ipc_open": (c_int32, [POINTER(c_uint8), POINTER(c_void_p)]),
    "dunet_ipc_close": (c_int32, [c_void_p]),
    "dunet_ipc_free": (c_int32, [c_void_p]),
    "dunet_q_sample": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int64, c_uint64, c_int64, c_void_p]),
    "dunet_dice_counts": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int64, c_void_p, c_void_p]),
    "dunet_hd95_workspace_bytes": (c_int32, [c_int32, POINTER(c_int32), POINTER(c_size_t)]),
    "dunet_hd95": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, POINTER(c_int32), POINTER(ctypes.c_double), c_void_p, c_void_p,
                             c_size_t, c_void_p]),
    "dunet_op_conv3x3x3": (c_int32, [c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32, POINTER(c_int32), c_int32, c_void_p]),
    "dunet_op_deconv2x2x2": (c_int32, [c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_void_p, c_int32, POINTER(c_int32), c_int32, c_void_p]),
    "dunet_debug_conv_geometry": (c_int32, [POINTER(c_int32), c_int32, c_int32, c_uint32, POINTER(c_int32)]),
    "dunet_debug_set_conv_timeline": (c_int32, [c_void_p]),
    "dunet_profile_enable": (c_int32, [c_void_p, c_int32]),
    "dunet_profile_read": (c_int32, [c_void_p, POINTER(ctypes.c_double), POINTER(c_uint64), POINTER(ctypes.c_double)]),
    "dunet_profile_read_all": (c_int32, [c_void_p, POINTER(ctypes.c_double), POINTER(c_uint64), POINTER(ctypes.c_double)]),
    "dunet_profile_dump": (c_int32, [c_void_p, POINTER(ctypes.c_double), POINTER(c_int32), c_int32, POINTER(c_int32)]),
    "dunet_debug_barrier_timeouts": (c_int32, [POINTER(c_uint32)]),
    "dunet_launch_count": (c_uint64, []),
}

_lib = None


def load(build_if_missing: bool = True) -> ctypes.CDLL:
    """Load the CUDA library, (re)building it in-tree with nvcc first when it is missing or older than its sources (the
    build is a no-op when the source digest matches the stamp; it is serialised across processes by a file lock and the
    .so is replaced atomically, so concurrent ranks never dlopen a half-written file).  Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing:
        import importlib.util

        spec = importlib.util.spec_from_file_location("_dunet_build", os.path.join(HERE, "build.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        try:
            mod.build()
        except Exception:
            if not os.path.exists(LIB_PATH):  # no compiler on this box: a prebuilt library (it travels with the tree) is fine
                raise
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing and there is no non-CUDA fallback; run diff-unet-amos_b200/build.py")
    lib = ctypes.CDLL(LIB_PATH)
    lib.dunet_version.restype = c_int32
    if lib.dunet_version() != DUNET_VERSION:  # e.g. a stale prebuilt library whose rebuild failed
        raise ImportError(f"{LIB_PATH} implements ABI version {lib.dunet_version()}, these bindings need {DUNET_VERSION}; "
                          "rebuild it with diff-unet-amos_b200/build.py")
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != 0:
        raise DunetError(code, load().dunet_last_error().decode("utf-8", "replace"))


def i32x3(v):
    return (c_int32 * 3)(int(v[0]), int(v[1]), int(v[2]))
