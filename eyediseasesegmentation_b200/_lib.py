"""ctypes binding of ``libeds_b200.so`` (see ``include/eds_b200.h``).

The shared library is the product; this module only declares prototypes and turns
error codes into exceptions.  There is deliberately no fallback: if the library is
missing or no sm_100 device is visible, compute entry points raise.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libeds_b200.so")

EDS_BF16, EDS_F32 = 0, 1
UP_NEAREST, UP_BILINEAR, UP_NONE = 0, 1, 2
PR_KEY_SHIFT = 14
PR_KEY_BIAS = (103 << 9) - 1
PR_HALF = 23 * 512 + 2
PR_BINS = 2 * PR_HALF
PR_NTHRESH = 19
STEM_PACKED_ELEMS = 64 * 184
#: thresholds of the reference's pooled PR / ROC curves (src/main/aucpr.py:53,128)
PR_THRESHOLDS = [0, 0.00001, 0.0001, 0.001, 0.01, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9,
                 0.99, 0.999, 0.9999, 0.99999, 1]

_vp, _i, _i64, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float


class GatedSrc(C.Structure):
    """``eds_gated_src`` of include/eds_b200.h."""
    _fields_ = [("x", C.c_void_p), ("cgate", C.c_void_p), ("sgate", C.c_void_p), ("C", C.c_int)]


# name -> argtypes; every function returns int except the two noted below.
PROTOTYPES = {
    "eds_version": [],
    "eds_device_ok": [],
    "eds_init": [],
    "eds_pr_hist_f32": [_vp, _vp, _i64, _i, _vp, _vp, _i, _vp],
    "eds_pr_hist_rects_f32": [_vp, _vp, _i, _i, _i, C.POINTER(_i), _vp, _vp, _vp],
    "eds_pr_scan": [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp],
    "eds_confusion_u8": [_vp, _vp, _i64, _i, _i, _i, _vp, _vp],
    "eds_tta_merge": [_vp, _i, _i, _i, C.POINTER(_i), _i, _vp, _vp],
    "eds_resize_paste_f32": [_vp, _i, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "eds_paste_tiles_x2_f32": [_vp, _i, _i, C.POINTER(_i), C.POINTER(_i), _vp, _i, _i, _vp],
    "eds_paste_tiles_owned_x2_f32": [_vp, _i, _i, _i, _i, C.POINTER(_i), C.POINTER(_i), _vp, _i, _i, _vp],
    "eds_tta_blend_supported": [_i, _i, C.POINTER(_i), _i],
    "eds_tta_blend_x2_f32": [_vp, _i, _i, _i, _i, _i, C.POINTER(_i), _i, _i, C.POINTER(_i), C.POINTER(_i), _vp, _i, _i, _vp],
    "eds_blend_tile_gaussian_x2_f32": [_vp, _i, _i, _i, _vp, _vp, _vp, _i, _i, _vp],
    "eds_blend_finalize_f32": [_vp, _vp, _i64, _vp, _vp],
    "eds_preprocess_tile_u8": [_vp, _i, _i, _i, _i, _i, C.POINTER(C.c_double), C.POINTER(C.c_double), _vp, _vp],
    "eds_stem_conv7x7s2": [_vp, _i, _i, _i, _i, C.POINTER(_i), _vp, _vp, _vp, _i, _vp],
    "eds_stem_pack_weights": [_vp, _vp, _vp],
    "eds_stem_conv7x7s2_mma": [_vp, _i, _i, _i, _i, C.POINTER(_i), _vp, _vp, _vp, _vp],
    "eds_conv2d_igemm_bf16": [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    "eds_conv2d_igemm_bf16_gated": [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    "eds_conv2d_igemm_grouped_supported": [_i, _i, _i, _i, _i, _i],
    "eds_conv2d_igemm_bf16_grouped": [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    "eds_affine_rows": [_vp, _i, _i, _vp, _vp, _i, _vp, _vp],
    "eds_conv3x3_halo_supported": [_i, _i, _i, _i, _i, _i],
    "eds_conv3x3_halo_bf16": [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp],
    "eds_conv3x3_small_supported": [_i, _i],
    "eds_conv3x3_small_bf16": [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp],
    "eds_conv2d_simt": [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp],
    "eds_conv2d_simt_grouped": [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp],
    "eds_head_conv3x3": [_vp, _i, _i, _i, _i, _vp, _vp, _i, _vp, _i, _vp],
    "eds_maxpool2d": [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _vp],
    "eds_avgpool2_affine": [_vp, _i, _i, _i, _i, _vp, _vp, _i, _vp, _i, _vp],
    "eds_channel_mean": [_vp, _i, _i, _i, _vp, _i, _vp],
    "eds_se_gate": [_vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "eds_se_scale_add_relu": [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _vp],
    "eds_upsample2x_concat": [_vp, _i, _i, _i, _i, _i, C.POINTER(_vp), C.POINTER(_i), _i, _vp, _i, _vp],
    "eds_gated_stats": [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp, _i, _i, _vp],
    "eds_gated_stats_multi": [_vp, _vp, _vp, _i, _i, _i, _i, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i), C.POINTER(_i),
                              C.POINTER(_vp), _i, _vp],
    "eds_sse_finalize": [_vp, _vp, _i, _i, _i, _i, _f, _vp, _vp],
    "eds_concat_gated": [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i, _vp],
    "eds_concat_gated_split": [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp],
    "eds_conv2d_igemm_bf16_2src": [_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    "eds_conv3x3_halo_bf16_2src": [_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp],
    "eds_conv3x3_wide_supported": [_i, _i, _i, _i, _i, _i],
    "eds_conv3x3_wide_bf16": [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp],
    "eds_conv3x3_wide_bf16_2src": [_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp],
    "eds_apply_gate": [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _vp],
    "eds_axial_attention": [_vp, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp],
    "eds_mhca_gate": [_vp, _vp, _i, _i, _i, _i, _vp, _i, _vp],
    "eds_cast_f32_to_bf16": [_vp, _vp, _i64, _vp],
    "eds_cast_bf16_to_f32": [_vp, _vp, _i64, _vp],
}
EXPORTS = sorted(list(PROTOTYPES) + ["eds_last_error"])

_lock = threading.Lock()
_lib = None
_inited = False


class EdsError(RuntimeError):
    """A libeds_b200 entry point returned a negative status."""


def load() -> C.CDLL:
    """dlopen the library and attach prototypes (no CUDA call is made)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise ImportError(
                    f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                    "or `make -C eyediseasesegmentation_b200/csrc`.  There is no CPU or PyTorch fallback.")
            lib = C.CDLL(LIB_PATH)
            for name, argtypes in PROTOTYPES.items():
                fn = getattr(lib, name)
                fn.argtypes = argtypes
                fn.restype = C.c_int
            lib.eds_last_error.argtypes = []
            lib.eds_last_error.restype = C.c_char_p
            _lib = lib
    return _lib


def lib() -> C.CDLL:
    """Library handle with the one-time device initialisation done; raises without a B200."""
    global _inited
    handle = load()
    if not _inited:
        rc = handle.eds_init()
        if rc != 0:
            raise EdsError(f"eds_init failed ({rc}): {handle.eds_last_error().decode()}")
        _inited = True
    return handle


def check(rc: int) -> None:
    if rc != 0:
        raise EdsError(f"libeds_b200 error {rc}: {load().eds_last_error().decode()}")


def int_array(values):
    arr = (C.c_int * len(values))(*[int(v) for v in values])
    return arr
