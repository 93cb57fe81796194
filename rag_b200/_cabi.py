"""ctypes binding of librag_b200.so (the C ABI declared in include/rag_b200.h).

The library is loaded once at module scope so that nn.Modules never hold ctypes handles (they
must stay deepcopy/pickle-safe: src/approaches/rag.py:225, src/utils.py:64-70 of the reference).
There is NO fallback: if the library is missing it is built with nvcc; if that fails, or a call
returns non-zero, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

ABI_VERSION = 17

_f = C.POINTER(C.c_float)
_d = C.POINTER(C.c_double)
_u8 = C.POINTER(C.c_uint8)
_i = C.c_int
_vp = C.c_void_p

# name -> (restype, argtypes); must list every symbol include/rag_b200.h declares
SIGNATURES = {
    "rag_abi_version": (_i, []),
    "rag_last_error": (C.c_char_p, []),
    "rag_launch_count": (C.c_uint64, []),
    "rag_cost_volume_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "rag_cost_volume_bwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "rag_disp_head_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "rag_disp_head_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "rag_disparity_regression_fwd": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "rag_disparity_regression_bwd": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "rag_upsample_trilinear": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_cost_volume_fwd_ws": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "rag_cost_volume_fwd_v": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "rag_cost_volume_bwd_v": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_disp_head_fwd_v": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_disp_head_bwd_v": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_loss_metrics_scratch": (_i, [_i, _i]),
    "rag_loss_metrics_sums": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, C.c_float, _vp]),
    "rag_smooth_l1_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, C.c_float, _vp]),
    "rag_cv_stem_workspace_bytes": (C.c_size_t, [_i, _i]),
    "rag_cv_stem_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "rag_cv_stem_fwd_v": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "rag_cv_stem_moments": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "rag_bn3d_moments": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "rag_bn3d_finalize": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, C.c_double, C.c_double, C.c_double, _i, _i, _vp]),
    "rag_bn3d_relu": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "rag_bn3d_bwd_sums": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "rag_bn3d_bwd_consts": (_i, [_vp, _vp, _vp, _vp, _i, C.c_double, _i, _vp]),
    "rag_bn3d_bwd_gz": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "rag_cv_stem_bwd_workspace_bytes": (C.c_size_t, [_i, _i, _i, _i, _i]),
    "rag_cv_stem_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_conv3d_c1_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "rag_conv3d_c1_bwd_workspace_bytes": (C.c_size_t, [_i]),
    "rag_conv3d_c1_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "rag_conv3d_cc_fwd": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_conv3d_cc_bwd_workspace_bytes": (C.c_size_t, [_i, _i, _i, _i, _i, _i]),
    "rag_conv3d_cc_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_conv3d_pw_fwd": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_conv3d_pw_bwd_workspace_bytes": (C.c_size_t, [_i, _i, _i, _i, _i, _i]),
    "rag_conv3d_pw_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_trilinear_resize_fwd": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_trilinear_resize_bwd": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_bilinear_resize_fwd": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_bilinear_resize_bwd": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_grid_sample_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_grid_sample_bwd_workspace_bytes": (C.c_size_t, [_i, _i, _i, _i, _i, _i]),
    "rag_grid_sample_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_size_t, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "rag_normalize_pad": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
}

LIB_PATH = _build.LIB
_lib = None


def lib() -> C.CDLL:
    """Load (building first if the .so is absent or stale) and type the library."""
    global _lib
    if _lib is not None:
        return _lib
    if _build.needs_build():
        _build.build()
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing and could not be built; rag_b200 has no fallback path")
    handle = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    got = handle.rag_abi_version()
    if got != ABI_VERSION:
        raise RuntimeError(f"librag_b200.so ABI version {got} != binding version {ABI_VERSION}; rebuild with python -m rag_b200.build")
    _lib = handle
    return _lib


def check(code: int, what: str) -> None:
    if code != 0:
        msg = lib().rag_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed with code {code}: {msg}")


def launch_count() -> int:
    return int(lib().rag_launch_count())
