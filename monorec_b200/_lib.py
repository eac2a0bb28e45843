"""ctypes binding of libmonorec_b200.so (the C ABI declared in include/monorec_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, an exception is raised.
"""
import ctypes
from ctypes import c_char_p, c_float, c_int, c_longlong, c_void_p, POINTER
from pathlib import Path

import os

_PKG = Path(__file__).resolve().parent
# MONOREC_B200_LIB: load another build of the library (kernel-variant experiments: tools/build_variant.py)
LIB_PATH = Path(os.environ["MONOREC_B200_LIB"]) if os.environ.get("MONOREC_B200_LIB") else _PKG / "libmonorec_b200.so"
_lib = None

c_float_p = POINTER(c_float)

# name -> (restype, argtypes); mirrors include/monorec_b200.h one to one (tests/test_capi_symbols.py checks it)
SIGNATURES = {
    "mr_version": (c_int, []),
    "mr_last_error": (c_char_p, []),
    "mr_launch_count": (c_longlong, [c_int]),
    "mr_projection_tables": (c_int, [c_void_p, c_void_p, POINTER(c_void_p), POINTER(c_void_p), c_int, c_int, c_int,
                                     c_int, c_void_p, c_void_p, c_int, c_float, c_float, c_void_p]),
    "mr_cost_volume_fwd": (c_int, [c_void_p, POINTER(c_void_p), c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                   c_int, c_int, c_int, c_float, c_float_p, c_void_p]),
    "mr_cost_volume_fwd_gather": (c_int, [c_void_p, POINTER(c_void_p), c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                          c_int, c_int, c_int, c_int, c_float, c_float_p, c_void_p]),
    "mr_cost_volume_fwd_nhwc": (c_int, [c_void_p, POINTER(c_void_p), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                        c_int, c_int, c_int, c_int, c_int, c_float, c_float_p, c_void_p]),
    "mr_cost_volume_host_workspace": (c_longlong, [c_int, c_int, c_int, c_int, c_int]),
    "mr_cost_volume_host_sfcv_offset": (c_longlong, [c_int, c_int, c_int, c_int, c_int]),
    "mr_cost_volume_host": (c_int, [c_void_p] * 8 + [c_int] * 5 + [c_float] * 3 + [c_void_p, c_longlong]),
    "mr_conv2d_nhwc": (c_int, [c_void_p, c_void_p]),
    "mr_sizeof_conv_desc": (c_int, []),
    "mr_pack_conv_weights_bytes": (c_longlong, [c_int, c_int, POINTER(c_int), c_int, c_int, c_int, POINTER(c_int), POINTER(c_int)]),
    "mr_pack_conv_weights": (c_int, [c_void_p, c_int, c_int, POINTER(c_int), c_int, c_int, c_int, c_void_p]),
    "mr_subpixel_convt_k4s2": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, POINTER(c_int), POINTER(c_int)]),
    "mr_subpixel_upconv2": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, POINTER(c_int), POINTER(c_int)]),
    "mr_conv_workspace_bytes": (c_longlong, [c_void_p]),
    "mr_conv2d_nhwc_tc": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p]),
    "mr_conv2d_nhwc_tc_phases": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "mr_conv2d_nhwc_tc_plan": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mr_nchw_to_nhwc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "mr_nchw_to_nhwc_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "mr_maxpool2_nhwc_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "mr_max_over_frames_f16": (c_int, [c_void_p, c_void_p, c_int, c_longlong, c_void_p]),
    "mr_pool_and_frame_max": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mr_maxpool3s2_nhwc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mr_cast_f32_to_f16": (c_int, [c_void_p, c_void_p, c_longlong, c_void_p]),
    "mr_maxpool2_nhwc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "mr_max_over_frames": (c_int, [c_void_p, c_void_p, c_int, c_longlong, c_void_p]),
    "mr_sparse_metrics_workspace": (c_longlong, [c_int]),
    "mr_sparse_metrics": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, POINTER(c_int), c_float, c_int, c_void_p,
                                  c_void_p, c_longlong, c_void_p]),
    "mr_images_u8_to_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mr_pointcloud_keep_mask": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "mr_pointcloud_workspace": (c_longlong, [c_int, c_int, c_int]),
    "mr_pointcloud_add": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, POINTER(c_void_p), c_int, c_int, c_int, c_int, c_int,
                                  c_float, c_float, POINTER(c_int), c_void_p, c_float, c_void_p, c_longlong, c_longlong, c_void_p,
                                  c_void_p, c_longlong, c_void_p]),
    "mr_reprojection_loss_fwd": (c_int, [c_void_p, POINTER(c_void_p), c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                         c_void_p, c_void_p, c_void_p]),
    "mr_reprojection_loss_bwd": (c_int, [c_void_p, POINTER(c_void_p), c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                         c_int, c_void_p, c_void_p]),
    "mr_mask_volume": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
}


class MonorecLibraryError(RuntimeError):
    pass


def load(build_if_missing=True):
    """Returns the loaded CDLL.  Builds it in-tree with nvcc if absent and a compiler is available."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing and not os.environ.get("MONOREC_B200_LIB"):
        # no-op when the source digest matches the stamp; rebuilds a stale library (sources newer than the .so)
        from . import build as _build
        _build.build()
    if not LIB_PATH.exists():
        raise MonorecLibraryError(f"{LIB_PATH} not found: run `python -m monorec_b200.build` (needs nvcc, sm_100a)")
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().mr_last_error().decode(errors="replace")
        raise MonorecLibraryError(f"{what} failed (code {rc}): {msg}")


def ptr_array(tensors):
    """Host array of device (or host) pointers for the `const float* const*` parameters."""
    arr = (c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr


def launch_count(reset=False):
    return int(load().mr_launch_count(1 if reset else 0))
