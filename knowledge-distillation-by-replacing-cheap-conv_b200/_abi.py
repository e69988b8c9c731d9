"""ctypes binding of libkdcc.so (C ABI declared in include/kdcc.h).

The library is the product: if it is missing or a call fails this module raises -- there is no
PyTorch/CPU fallback anywhere in the package.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KDCC_LIB", os.path.join(_HERE, "libkdcc.so"))  # KDCC_LIB: A/B builds of the same library (tools/)

F32, BF16 = 0, 1
F32_TF32X3 = 2   # pointwise only: fp32 tensors, products as three tf32 tensor-core MMAs
NHWC, NCHW = 0, 1
PLANES_TO_NHWC = 2   # pointwise only: input / input-gradient as channel planes, output / output-gradient channels_last

_vp, _i, _l, _f, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_long, ctypes.c_float, ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/kdcc.h one to one
SIGNATURES = {
    "kdcc_version": (_i, []),
    "kdcc_strerror": (ctypes.c_char_p, [_i]),
    "kdcc_last_driver_status": (_i, []),
    "kdcc_dispatch_name": (ctypes.c_char_p, [_i] * 11),
    "kdcc_dw_fwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "kdcc_dw_bwd_workspace_bytes": (_sz, [_i] * 9),
    "kdcc_dw_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "kdcc_pw_fwd": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp, _l, _i, _i, _i, _i, _i, _vp]),
    "kdcc_pw_fwd_residual": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _l, _i, _i, _i, _i, _i, _vp]),
    "kdcc_pw_bwd_workspace_bytes": (_sz, [_i, _l, _i, _i, _i]),
    "kdcc_pw_bwd_dx": (_i, [_vp, _vp, _vp, _vp, _sz, _l, _i, _i, _i, _i, _i, _vp]),
    "kdcc_pw_bwd_dw": (_i, [_vp, _vp, _vp, _vp, _sz, _l, _i, _i, _i, _i, _i, _vp]),
    "kdcc_loss_workspace_bytes": (_sz, []),
    "kdcc_kd_loss": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _i, _i, _l, _l, _l, _l, _f, _i, _i, _f, _vp]),
    "kdcc_kd_loss_multi": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _sz, _i, _i, _l, _l, _l, _l, _f, _i, _f, _vp]),
    "kdcc_hint_loss": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _sz, _i, _i, _l, _i, _f, _i, _f, _vp]),
    "kdcc_ce_workspace_bytes": (_sz, [_i, _l]),
    "kdcc_ce_loss": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _sz, _i, _i, _l, _l, _l, _l, _i, _f, _vp]),
    "kdcc_logits_stats": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _f, _f, _vp, _vp, _vp, _vp, _vp, _sz, _i, _i, _l, _l, _l, _l,
                               _i, _vp]),
    "kdcc_ensemble_loss": (_i, [_vp, _vp, _vp, _i, _f, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _sz, _i, _i, _l, _l, _l, _l,
                                _i, _f, _f, _vp, _vp]),
    "kdcc_cast_f32_to_bf16": (_i, [_vp, _vp, _l, _vp]),
    "kdcc_scale_inplace": (_i, [_vp, _vp, _l, _i, _vp]),
    "kdcc_scale_inplace_expect": (_i, [_vp, _vp, _f, _l, _i, _vp]),
    "kdcc_layout_convert": (_i, [_vp, _vp, _i, _i, _l, _i, _i, _vp]),
    "kdcc_colsum": (_i, [_vp, _vp, _vp, _sz, _l, _i, _i, _vp]),
    "kdcc_colsum_workspace_bytes": (_sz, [_l, _i]),
    "kdcc_confusion_update": (_i, [_vp, _vp, _vp, _i, _i, _l, _l, _l, _i, _i, _vp]),
    "kdcc_radam_step": (_i, [_vp, _vp, _vp, _vp, _vp, _l, _f, _f, _f, _f, _f, _f, _f, _i, _vp]),
    "kdcc_radam_step_multi": (_i, [_vp, _vp, _l, _i, _vp, _vp, _vp, _l, _f, _f, _f, _f, _f, _f, _f, _i, _vp]),
    "kdcc_tta_stitch": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp, _i, _vp]),
    "kdcc_resize_bilinear": (_i, [_vp, _i, _i, _i, _vp, _i, _i, _f, _i, _vp]),
    "kdcc_tta_windows_workspace_bytes": (_sz, [_i] * 4),
    "kdcc_tta_windows": (_i, [_vp] + [_i] * 7 + [_f] * 6 + [_vp, _vp, _sz, _vp]),
    "kdcc_canny_workspace_bytes": (_sz, [_i, _i, _i]),
    "kdcc_canny": (_i, [_vp, _vp, _vp, _sz, _i, _i, _i, _i, _i, _i, ctypes.c_double, ctypes.c_double, _vp]),
}

_lib = None


class KdccError(RuntimeError):
    pass


def lib():
    """Load libkdcc.so (once).  Raises if it has not been built: there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise KdccError(
                "libkdcc.so not found at %s -- build it with `python __graft_entry__.py` "
                "(or knowledge-distillation-by-replacing-cheap-conv_b200/build.py); kdcc has no CPU/PyTorch fallback" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def strerror(code):
    return lib().kdcc_strerror(int(code)).decode()


def check(code, what):
    if code != 0:
        extra = ""
        if code == -2 and lib().kdcc_last_driver_status() != 0:
            extra = " [TMA descriptor encode returned CUresult %d]" % lib().kdcc_last_driver_status()
        raise KdccError("%s failed: %s (code %d)%s" % (what, strerror(code), code, extra))


def dispatch_name(op, N, H, W, C, Cout, k, dil, pad, layout, dtype):
    return lib().kdcc_dispatch_name(op, N, H, W, C, Cout, k, dil, pad, layout, dtype).decode()
