"""ctypes binding of the C-ABI library (include/kdme_b200.h).

The product path has no CPU fallback: if the CUDA library is missing this module
raises, and every operator raises on a non-zero status from the library.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# KDME_LIB_PATH: A/B runs of two builds of the library on the same GPU box (development only)
LIB_PATH = os.environ.get("KDME_LIB_PATH") or os.path.join(_HERE, "libkdme_b200.so")

KDME_OK = 0
KDME_EINVAL = -100001
KDME_ENOTSUP = -100002
KDME_MAX_RADIUS = 15
KDME_GUIDE_GRAY, KDME_GUIDE_BGR, KDME_GUIDE_BGRX = 1, 3, 4


class KdmeError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"kdme_b200 error {code}: {msg}")
        self.code = code


def build(verbose: bool = False) -> str:
    """Compile csrc/ for sm_100a (nvcc cross-compiles without a GPU)."""
    res = subprocess.run(["make", "-C", os.path.join(_HERE, "csrc")], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc build failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stdout)
    return LIB_PATH


_lib = None

# name -> (restype, argtypes); every symbol include/kdme_b200.h declares
_vp, _sz, _i, _f = C.c_void_p, C.c_size_t, C.c_int, C.c_float
SIGNATURES = {
    "kdme_last_error": (C.c_char_p, []),
    "kdme_version": (C.c_char_p, []),
    "jbf_create": (_i, [C.POINTER(_vp), _i, _i, _f, _f, _f, _i, _i, _i, _vp]),
    "jbf_destroy": (None, [_vp]),
    "jbf_set_presmooth": (_i, [_vp, _i, _f, _f]),
    "jbf_set_guide_channels": (_i, [_vp, _i]),
    "jbf_process": (_i, [_vp, _vp, _vp, _sz]),
    "jbf_process_xyz": (_i, [_vp, _vp, _vp, _sz, _vp, _f, _f, _i, _i]),
    "jbf_refine_stats": (_i, [_vp, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]),
    "jbf_process_batch": (_i, [_vp, _vp, _vp, _sz, _vp, _i]),
    "jbf_filter_guide4": (_i, [_vp, _vp, _vp, _sz, _vp, _i]),
    "jbf_presmooth": (_i, [_vp, _vp, _sz, _vp, _sz, _i]),
    "jbf_process_host": (_i, [_vp, _vp, _vp, _sz, _vp, _i]),
    "jbf_process_host_u16": (_i, [_vp, _vp, _vp, _sz, _vp, _i]),
    "kdme_host_alloc": (_vp, [_sz, _i]),
    "kdme_host_free": (None, [_vp]),
    "jbf_presmooth_rows": (_i, [_vp, _vp, _sz, _vp, _sz, _i]),
    "jbf_filter_rows": (_i, [_vp, _vp, _vp, _sz, _vp, _i, _i, _i]),
    "jbf_presmooth_rows_p2p": (_i, [_vp, _vp, _sz, _vp, _sz, _i, _i, _i, _vp, _vp]),
    "jbf_filter_rows_p2p": (_i, [_vp, _vp, _vp, _sz, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "jbf_filtered_device": (_vp, [_vp]),
    "jbf_filtered_host": (_vp, [_vp]),
    "jbf_smooth_device": (_vp, [_vp, C.POINTER(_sz)]),
    "jbf_guide4_device": (_vp, [_vp, C.POINTER(_sz)]),
    "jbf_upsample": (_i, [_vp, _vp, _i, _i, _vp, _sz, _vp]),
    "jbf_upsample_batch": (_i, [_vp, _vp, _i, _i, _vp, _sz, _vp, _i]),
    "jbf_upsample_batch_u16": (_i, [_vp, _vp, _i, _i, _vp, _sz, _vp, _i]),
    "jbf_kernel_variant": (_i, [_vp]),
    "jbf_mrf": (_i, [_vp, _vp, _vp, _sz, _vp, _i, _f, _f]),
    "kdme_projective_to_real": (_i, [_vp, _vp, _i, _i, _f, _f, _i, _i, _vp]),
    "kdme_depth_bilateral_xyz": (_i, [_vp, _vp, _vp, _i, _i, _i, _f, _f, _vp]),
    "kdme_mean_3d_error": (_i, [_vp, _vp, C.c_longlong, C.POINTER(C.c_double), C.POINTER(C.c_longlong), _vp]),
    "kdme_guided_upsample": (_i, [_vp, _i, _i, _vp, _vp, _sz, _vp, _i, _i, _i, _f, _f, _f, _vp]),
    "kdme_guided_fill": (_i, [_vp, _vp, _vp, _sz, _vp, _i, _i, _i, _f, _f, _f, _vp]),
    "kdme_guided_upsample_ex": (_i, [_vp, _i, _i, _vp, _vp, _sz, _i, _vp, _i, _i, _i, _f, _f, _f, _vp]),
    "kdme_guided_fill_ex": (_i, [_vp, _vp, _vp, _sz, _i, _vp, _i, _i, _i, _f, _f, _f, _vp]),
    "kdme_guided_fill_batch": (_i, [_vp, _vp, _vp, _sz, _i, _vp, _i, _i, _i, _i, _f, _f, _f, _vp]),
    "kdme_guided_fill_batch_u16": (_i, [_vp, _vp, _vp, _sz, _i, _vp, _i, _i, _i, _i, _f, _f, _f, _vp]),
    "kdme_guided_upsample_batch": (_i, [_vp, _i, _i, _vp, _vp, _sz, _i, _vp, _i, _i, _i, _i, _f, _f, _f, _vp]),
    "kdme_guided_upsample_batch_u16": (_i, [_vp, _i, _i, _vp, _vp, _sz, _i, _vp, _i, _i, _i, _i, _f, _f, _f, _vp]),
    "buf2d_create": (_i, [C.POINTER(_vp), _i, _i, _i, _vp]),
    "buf2d_destroy": (None, [_vp]),
    "buf2d_init": (_i, [_vp]),
    "buf2d_insert_f32": (_i, [_vp, _vp]),
    "buf2d_insert_dw": (_i, [_vp, _vp]),
    "buf2d_insert_f32x2": (_i, [_vp, _vp]),
    "buf2d_update_f32": (_i, [_vp, _vp]),
    "buf2d_update_batch_f32": (_i, [_vp, _vp, _i]),
    "buf2d_update_u16_host": (_i, [_vp, _vp]),
    "buf2d_get_depth": (_i, [_vp, _vp]),
    "buf2d_get_weight": (_i, [_vp, _vp]),
    "buf2d_raw": (_vp, [_vp]),
}


def lib():
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise FileNotFoundError(
                f"{LIB_PATH} is missing: build it with `make -C kinectdepthmapenhancement_b200/csrc` "
                "(or __graft_entry__.build()). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code: int) -> None:
    if code != KDME_OK:
        raise KdmeError(code, lib().kdme_last_error().decode("utf-8", "replace"))
