"""ctypes binding of libbacs_b200.so (include/bacs_b200.h).  No torch types cross the ABI:
only raw device pointers, sizes and the CUDA stream handle.

There is no fallback: if the library is missing, importing a symbol raises."""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libbacs_b200.so")

F32, BF16, F16 = 0, 1, 2
PIX_WEIGHTED_CE, PIX_CE, PIX_UNBIASED_CE, PIX_SCORE = 0, 1, 2, 3
ACC_LOSS, ACC_WSUM, ACC_FOCAL, ACC_KEPT, ACC_BG, ACC_INVALID, ACC_DISTILL_PIX, ACC_VALID = range(8)
NACC = 8

vp, i32, i64, f32, sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t


class PixelArgs(C.Structure):
    """struct bacs_pixel_args"""
    _fields_ = [
        ("logits", vp), ("labels", vp), ("dlogits", vp), ("preds", vp), ("z", vp), ("seen_max", vp), ("distill_mask", vp),
        ("gz", vp), ("class_w", vp), ("hist", vp), ("acc", vp), ("score", vp),
        ("B", i32), ("K", i32), ("H", i32), ("W", i32), ("T", i32), ("h", i32), ("w", i32),
        ("dtype", i32), ("mode", i32), ("old_cl", i32), ("ukd", i32), ("focal_head", i32),
        ("ignore_index", i32), ("seen_scale", i32),
        ("gamma", f32), ("threshold", f32), ("focal_gamma", f32), ("focal_alpha", f32),
        ("lkd_threshold", f32), ("grad_scale", f32),
        ("ready", vp), ("focal_scale_out", vp), ("loss_out", vp),
        ("focal_weight", f32), ("loss_coef", f32), ("loss_over_wsum", i32),
    ]


_SIGNATURES = {
    "bacs_version": (i32, []),
    "bacs_last_error_string": (C.c_char_p, []),
    "bacs_device_sm_count": (i32, []),
    "bacs_launch_count": (C.c_ulonglong, []),
    "bacs_label_hist": (i32, [vp, i64, vp, vp]),
    "bacs_label_remap_workspace_bytes": (sz, [i64]),
    "bacs_label_remap": (i32, [vp, vp, i64, i64, i32, i32, vp, i32, vp, i32, vp, vp]),
    "bacs_label_downsample_task": (i32, [vp, i32, i32, i32, i32, i32, vp, i32, vp, vp, vp, vp, vp]),
    "bacs_proto_workspace_bytes": (sz, [i32, i32, i32]),
    "bacs_proto_accumulate": (i32, [vp, i32, i32, i32, i32, i32, vp, vp, vp, i32, i32, vp, vp, vp, sz, vp]),
    "bacs_proto_accumulate_update": (i32, [vp, i32, i32, i32, i32, i32, vp, vp, vp, i32, i32, vp, vp, vp, sz, vp, vp, i32,
                                           vp, vp]),
    "bacs_proto_update": (i32, [vp, vp, i32, vp, vp, i32, i32, vp, vp]),
    "bacs_seen_logits": (i32, [vp, i32, i32, i32, i32, i32, vp, vp, vp, i32, vp, vp]),
    "bacs_seen_logits_heads": (i32, [vp, i32, i32, i32, i32, i32, vp, vp, vp, i32, vp, vp, vp]),
    "bacs_seen_upsample": (i32, [vp, i32, i32, i32, i32, i32, i32, vp, vp]),
    "bacs_seen_head_backward": (i32, [vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]),
    "bacs_focal_scale": (i32, [vp, vp, f32, vp, vp, vp]),
    "bacs_focal_scale_loss": (i32, [vp, vp, f32, f32, i32, vp, vp, vp]),
    "bacs_pixel_workspace_bytes": (sz, [C.POINTER(PixelArgs)]),
    "bacs_pixel_kernel_variant": (i32, [C.POINTER(PixelArgs)]),
    "bacs_pixel_loss": (i32, [C.POINTER(PixelArgs), vp, sz, vp]),
    "bacs_pixel_lowres_workspace_bytes": (sz, [C.POINTER(PixelArgs), i32, i32]),
    "bacs_pixel_loss_lowres": (i32, [C.POINTER(PixelArgs), i32, i32, vp, sz, vp]),
    "bacs_pseudo_label": (i32, [vp, i32, i32, i32, i32, i32, vp, vp]),
    "bacs_pseudo_label_lowres": (i32, [vp, i32, i32, i32, i32, i32, i32, i32, vp, vp]),
    "bacs_distill_workspace_bytes": (sz, [i32, i32, i32, i32, i32, i32]),
    "bacs_teacher_distill": (i32, [vp, vp, i32, i32, i32, i32, i32, vp, i32, i32, f32, vp, vp, vp, vp, sz, vp]),
    "bacs_teacher_distill_add": (i32, [vp, vp, i32, i32, i32, i32, i32, vp, i32, i32, f32, vp, vp, vp, vp, vp, sz, vp]),
    "bacs_distill_set_mode": (i32, [i32]),
    "bacs_distill_kernel_variant": (i32, [i32, i32, i32, i32, i32, i32, i32]),
    "bacs_der_workspace_bytes": (sz, [i32, i32, i32]),
    "bacs_der_mse": (i32, [vp, i32, vp, i32, i32, vp, i32, i32, i32, i32, f32, vp, vp, vp, sz, vp]),
    "bacs_unbiased_kd_workspace_bytes": (sz, [i64]),
    "bacs_unbiased_kd": (i32, [vp, vp, i32, i32, i32, i32, i32, i32, f32, vp, f32, vp, vp, vp, sz, vp]),
    "bacs_der_cut": (i32, [vp, i32, i32, vp, vp]),
    "bacs_confmat_accumulate": (i32, [vp, i32, vp, i64, i32, vp, vp, vp]),
    "bacs_confmat_metrics": (i32, [vp, i32, vp, vp]),
    "bacs_class_distance_workspace_bytes": (sz, [i32, i32, i32, i32, i32]),
    "bacs_class_distance": (i32, [vp, i32, i32, i32, i32, i32, vp, i32, vp, vp, vp, sz, vp]),
    "bacs_class_sums_workspace_bytes": (sz, [i32, i32, i32]),
    "bacs_class_sums": (i32, [vp, i32, i32, i32, i32, i32, vp, i32, vp, vp, sz, vp]),
    "bacs_gather_rows": (i32, [vp, i64, i64, vp, i64, vp, vp]),
    "bacs_scale_inplace": (i32, [vp, i32, i64, vp, vp]),
    "bacs_scale_inplace_multi": (i32, [i32, C.POINTER(vp), C.POINTER(i32), C.POINTER(i64), vp, vp]),
    "bacs_peer_allreduce": (i32, [vp, i32, i32, i32, i32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), vp, vp, vp, vp, i32,
                                  i32, i32, vp, vp]),
    "bacs_peer_set_timeout_ms": (i32, [i64]),
    "bacs_pack_state": (i32, [vp, vp, i32, i32, vp, i32, vp, vp]),
    "bacs_unpack_state": (i32, [vp, i32, i32, vp, vp, vp, i32, vp]),
    "bacs_combine_scalars": (i32, [i32, C.POINTER(vp), C.POINTER(i32), C.POINTER(vp), C.POINTER(i32),
                                   C.POINTER(f32), vp, vp]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


class BacsError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Loads the library (once).  Raises if it has not been built -- never falls back."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BacsError(
                "libbacs_b200.so not found at %s: build it with `python -m bacs_b200.build` "
                "(there is no CPU / PyTorch fallback for the BACS loss path)" % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error() -> str:
    return load().bacs_last_error_string().decode("utf-8", "replace")


def check(status: int, what: str) -> None:
    if status != 0:
        raise BacsError("%s failed (status %d): %s" % (what, status, last_error()))
