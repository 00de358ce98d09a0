"""ctypes binding of libmte.so (the C ABI declared in include/mte.h).

There is NO fallback: if the library is missing or does not export a symbol the
import fails loudly.  PyTorch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MTE_LIB", os.path.join(_HERE, "libmte.so"))  # MTE_LIB: A/B builds while tuning

MTE_MAX_SCALES = 4
MTE_MAX_THRESHOLDS = 254
MTE_WS_HEADER_BYTES = 65536
MTE_F32, MTE_F64, MTE_U8 = 0, 1, 2
MTE_LOSS_CE, MTE_LOSS_ATTENTION, MTE_LOSS_SPATIAL, MTE_LOSS_DICE = 1, 2, 4, 8


class MteError(RuntimeError):
    pass


class LossScale(C.Structure):
    _fields_ = [
        ("pred", C.c_void_p), ("edge", C.c_void_p), ("normal", C.c_void_p), ("mask", C.c_void_p),
        ("grad_map", C.c_void_p), ("grad_pred", C.c_void_p), ("stash", C.c_void_p),
        ("B", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("scale_weight", C.c_float),
    ]


class LossAttrs(C.Structure):
    _fields_ = [
        ("is_grad", C.c_int32), ("is_sigmoid", C.c_int32), ("pred_is_inverse", C.c_int32),
        ("sigmoid_thresh", C.c_float), ("weight", C.c_float), ("pos_to_neg", C.c_float),
    ]


_vp, _sz, _i, _d = C.c_void_p, C.c_size_t, C.c_int, C.c_double
_SIGNATURES = {
    "mte_version": (C.c_int, []),
    "mte_error_string": (C.c_char_p, [_i]),
    "mte_workspace_init": (_i, [_vp, _sz, _vp]),
    "mte_edge_loss_workspace_bytes": (_sz, [C.POINTER(LossScale), _i]),
    "mte_edge_loss_ctx_bytes": (_sz, [C.POINTER(LossScale), _i]),
    "mte_edge_loss_fwd": (_i, [C.POINTER(LossScale), _i, C.POINTER(LossAttrs), _vp, _vp, _vp, _sz, _vp]),
    "mte_edge_loss_bwd": (_i, [C.POINTER(LossScale), _i, C.POINTER(LossAttrs), _vp, _vp, _vp, _sz, _vp]),
    "mte_edge_loss_fused_supported": (_i, [C.POINTER(LossScale), _i, C.POINTER(LossAttrs)]),
    "mte_edge_loss_fwd_grad": (_i, [C.POINTER(LossScale), _i, C.POINTER(LossAttrs), _vp, _vp, _vp, _vp, _sz, _vp]),
    "mte_edge_loss_grad_rescale": (_i, [C.POINTER(LossScale), _i, _vp, _vp, _vp, _vp]),
    "mte_canny_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "mte_canny_from_depth": (_i, [_vp, _i, _i, _i, _i, _d, _d, C.POINTER(C.c_int32), C.POINTER(C.c_int32), _i,
                                  _vp, _vp, _vp, _sz, _vp]),
    "mte_resize_linear": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    "mte_dee_workspace_bytes": (_sz, [_i, _i, _i]),
    "mte_dee_postprocess": (_i, [_vp, _i, _i, _i, _i, _i, _i, _d, _d, _vp, _vp, _i, _vp, _sz, _vp]),
    "mte_pr_workspace_bytes": (_sz, [_i, _i, _i, _i, _d]),
    "mte_pr_thin_workspace_bytes": (_sz, [_i, _i, _i, _i, _d]),
    "mte_pr_counts": (_i, [_vp, _i, _vp, _i, _i, _i, C.POINTER(C.c_int32), C.POINTER(C.c_double), _i, _d, _i,
                           _vp, _vp, _sz, _vp]),
    "mte_pr_counts_per_image": (_i, [_vp, _i, _vp, _i, _i, _i, C.POINTER(C.c_int32), C.POINTER(C.c_double), _i, _d,
                                     _i, _vp, _vp, _sz, _vp]),
    "mte_match_workspace_bytes": (_sz, [_i, _i, _i, _d]),
    "mte_correspond_pixels": (_i, [_vp, _vp, _i, _i, _i, _d, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mte_thin_workspace_bytes": (_sz, [_i, _i, _i]),
    "mte_binary_thin": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _sz, _vp]),
    "mte_edge_loss_alt_workspace_bytes": (_sz, [_i, _i, _i]),
    "mte_edge_loss_alt_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, C.c_float, C.c_float, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mte_edge_loss_alt_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, C.c_float, C.c_float, _vp, _vp,
                                   _vp, _i, _vp, _sz, _vp]),
    "mte_decode_normals": (_i, [_vp, _vp, _sz, _vp]),
    "mte_edge_resize_workspace_bytes": (_sz, [_i]),
    "mte_edge_resize_preserve": (_i, [_vp, _i, _i, _i, _vp, _i, _i, _vp, _sz, _vp]),
    "mte_chamfer_workspace_bytes": (_sz, [_i, _i, _i]),
    "mte_chamfer_counts": (_i, [_vp, _vp, _i, _i, _i, _d, _vp, _vp, _vp, _sz, _vp]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def _load():
    if not os.path.exists(LIB_PATH):
        raise MteError(
            f"{LIB_PATH} not found: build it with `python -m mindtheedge_b200.build` "
            "(there is no CPU or PyTorch fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise MteError(f"libmte.so does not export {name}") from exc
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(rc: int, what: str = "libmte call"):
    if rc != 0:
        raise MteError(f"{what} failed: {lib.mte_error_string(rc).decode()} (code {rc})")
