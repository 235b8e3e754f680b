"""ctypes binding of libclipk.so (the C ABI declared in include/clipk.h).

There is no fallback of any kind: if the shared library is missing or the device is not a B200-class GPU
(compute capability 10.x) the first compute call raises.  The library is built in-tree by
``megatron-clip_b200/build.py`` (nvcc, sm_100a) and lives next to this file.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libclipk.so")

BF16 = 0
F32 = 1
F16 = 3
F16X2 = 4

_ERRNAMES = {-1: "CLIPK_EINVAL", -2: "CLIPK_EUNSUPPORTED", -3: "CLIPK_EARCH", -4: "CLIPK_EWORKSPACE",
             -5: "CLIPK_EDRIVER"}

# name -> (restype, argtypes); mirrors include/clipk.h one to one
_vp, _i, _ll, _f, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_float, ctypes.c_size_t
PROTOTYPES = {
    "clipk_version": (_i, []),
    "clipk_launch_count": (_ll, []),
    "clipk_last_error": (ctypes.c_char_p, []),
    "clipk_check_device": (_i, []),
    "clipk_to_f16": (_i, [_vp, _i, _ll, _ll, _ll, _vp, _i, _ll, _vp, _vp]),
    "clipk_fwd_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "clipk_fwd_stats": (_i, [_vp, _vp, _i, _i, _i, _ll, _ll, _i, _vp, _vp, _vp, _ll, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "clipk_fwd_both_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "clipk_fwd_both": (_i, [_vp, _vp, _i, _i, _i, _ll, _ll, _i, _vp, _vp, _vp, _ll, _vp, _vp, _vp, _vp, _i, _vp, _sz, _vp]),
    "clipk_to_f16_amax": (_i, [_vp, _i, _ll, _ll, _ll, _vp, _i, _ll, _vp, _vp, _vp]),
    "clipk_finalize": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _ll, _i, _ll, _vp, _vp, _vp, _vp]),
    "clipk_bwd_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "clipk_bwd": (_i, [_vp, _vp, _i, _i, _i, _ll, _ll, _i, _vp, _vp, _vp, _vp, _ll, _ll, _i, _vp, _vp,
                       _vp, _ll, _vp, _vp, _f, _f, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "clipk_normalize_fwd": (_i, [_vp, _i, _ll, _ll, _ll, _vp, _ll, _vp, _f, _vp]),
    "clipk_normalize_bwd": (_i, [_vp, _ll, _vp, _ll, _vp, _i, _ll, _ll, _vp, _ll, _f, _vp]),
    "clipk_cast": (_i, [_vp, _vp, _ll, _i, _vp]),
    "clipk_debug_tmem_layout": (_i, [_vp, _vp]),
    "clipk_rank_count": (_i, [_vp, _i, _i, _ll, _vp, _ll, _ll, _vp, _vp, _vp]),
    "clipk_distill_cross": (_i, [_vp, _vp, _i, _i, _ll, _vp, _vp, _vp, _vp, _ll, _vp, _vp, _vp]),
    "clipk_distill_grad": (_i, [_vp, _vp, _i, _i, _ll, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _vp, _ll, _vp]),
    "clipk_gemm16": (_i, [_vp, _vp, _vp, _i, _i, _i, _ll, _ll, _ll, _i, _i, _i, _i, _vp]),
}


MAX_PEERS = 8
STAT_WORDS = 8


class Peer(ctypes.Structure):
    """struct clipk_peer (include/clipk.h)."""
    _fields_ = [("world", _i), ("rank", _i),
                ("text_src", _vp * MAX_PEERS), ("stats_src", _vp * MAX_PEERS), ("col_src", _vp * MAX_PEERS),
                ("grad_slot", _vp * MAX_PEERS), ("flags_gather", _vp * MAX_PEERS), ("flags_stats", _vp * MAX_PEERS),
                ("flags_grad", _vp * MAX_PEERS),
                ("epoch_gather", ctypes.c_uint), ("epoch_stats", ctypes.c_uint), ("epoch_grad", ctypes.c_uint),
                ("my_slots", _vp), ("err", _vp)]


class Step(ctypes.Structure):
    """struct clipk_step (include/clipk.h)."""
    _fields_ = [("rows", _i), ("cols", _i), ("d", _i), ("src_dtype", _i), ("normalize", _i), ("eps", _f),
                ("image", _vp), ("text", _vp), ("ld_image", _ll), ("ld_text", _ll), ("logit_scale", _vp),
                ("loss_div", _f), ("grad_coef", _f), ("grad_split", _i),
                ("x_op", _vp), ("y_all", _vp), ("inv_x", _vp), ("inv_y", _vp), ("stats", _vp), ("lse_row", _vp),
                ("lse_col", _vp), ("scal", _vp), ("g16", _vp),
                ("grad_out", _vp), ("d_image", _vp), ("d_text", _vp), ("d_scale", _vp), ("out_dtype", _i),
                ("peer", ctypes.POINTER(Peer)), ("workspace", _vp), ("workspace_bytes", _sz), ("stream", _vp)]


SIGLIP_STATE_WORDS = 8


class Siglip(ctypes.Structure):
    """struct clipk_siglip (include/clipk.h)."""
    _fields_ = [("rows", _i), ("cols", _i), ("d", _i), ("x", _vp), ("ldx", _ll), ("y", _vp), ("ldy", _ll),
                ("logit_scale", _vp), ("logit_bias", _vp), ("diag_offset", _ll), ("state", _vp),
                ("grad_out", _vp), ("d_x", _vp), ("d_y", _vp), ("d_scale", _vp), ("d_bias", _vp),
                ("workspace", _vp), ("workspace_bytes", _sz), ("stream", _vp)]


PROTOTYPES.update({
    "clipk_siglip_workspace_bytes": (_sz, [ctypes.POINTER(Siglip)]),
    "clipk_siglip_forward": (_i, [ctypes.POINTER(Siglip)]),
    "clipk_siglip_backward": (_i, [ctypes.POINTER(Siglip)]),
    "clipk_bwd_panel": (_i, [_i, _i, _i, ctypes.POINTER(_ll), ctypes.POINTER(_ll)]),
    "clipk_profile_begin": (_i, [_vp]),
    "clipk_profile_end": (_i, [ctypes.c_char_p, _sz]),
    "clipk_step_workspace_bytes": (_sz, [ctypes.POINTER(Step)]),
    "clipk_step_forward": (_i, [ctypes.POINTER(Step)]),
    "clipk_step_backward": (_i, [ctypes.POINTER(Step)]),
})


class ClipkError(RuntimeError):
    pass


_lib = None


def load():
    """Load libclipk.so once; raise ClipkError (never fall back) when it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ClipkError(
            f"{LIB_PATH} not found: build it with `python megatron-clip_b200/build.py` (nvcc, sm_100a). "
            "clipk has no CPU or non-Blackwell fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)   # AttributeError here means header and library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc == 0:
        return
    msg = load().clipk_last_error().decode(errors="replace")
    name = _ERRNAMES.get(rc, f"cudaError {rc}" if rc > 0 else str(rc))
    raise ClipkError(f"{what} failed: {name}: {msg}")
