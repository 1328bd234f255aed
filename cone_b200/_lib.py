"""ctypes binding of libcone_b200.so (include/cone_b200.h).  There is no fallback: if the library is
missing or a call fails, an exception is raised."""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcone_b200.so")

PREC_FP32 = 0
PREC_TC = 1
PREC_TC_SPLIT = 2  # cone_linear only: 3-product split-fp16 GEMM (fp32-class accuracy on the tensor pipe)

# storage type of a raw feature tensor passed to the _ex entry points
DTYPE_F32 = 0
DTYPE_F16 = 1
DTYPE_BF16 = 2

# include/cone_b200.h: most candidates per query of cone_fuse_nms(_ex) (shared memory) and of cone_fuse_nms_ws
FUSE_NMS_MAX_SHARED_CANDIDATES = 2201
FUSE_NMS_MAX_CANDIDATES = 131072


class ConeDims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("v_dim", "t_dim", "hidden", "nheads", "ffn", "enc_layers", "dec_layers",
                                         "num_queries", "max_v_l", "max_q_l", "m_dim")]


class ConeError(RuntimeError):
    pass


_lock = threading.Lock()
_lib = None

_p = C.c_void_p
_i32, _i64, _sz, _f32, _f64 = C.c_int32, C.c_int64, C.c_size_t, C.c_float, C.c_double

# name -> (restype, argtypes); mirrors include/cone_b200.h one to one
SIGNATURES = {
    "cone_last_error": (C.c_char_p, []),
    "cone_version": (C.c_int, []),
    "cone_weights_create": (C.c_int, [_p, _sz, C.POINTER(ConeDims), _p, C.POINTER(_p)]),
    "cone_weights_destroy": (None, [_p]),
    "cone_weights_update": (C.c_int, [_p, _p, _sz, _p]),
    "cone_weights_expected_floats": (_sz, [C.POINTER(ConeDims)]),
    "cone_workspace_bytes": (_sz, [C.POINTER(ConeDims), _i64, _i32, _i32]),
    "cone_prepare_workspace_bytes": (_sz, [C.POINTER(ConeDims), _i64]),
    "cone_l2_normalize": (C.c_int, [_p, _p, _i64, _i32, _f32, _p]),
    "cone_l2_normalize_ex": (C.c_int, [_p, _i32, _p, _i64, _i32, _f32, _p]),
    "cone_video_prepare": (C.c_int, [_p, _p, _i64, _p, _p, _p, _sz, C.c_int, _p]),
    "cone_video_prepare_ex": (C.c_int, [_p, _p, _i32, _i64, _p, _p, _p, _sz, C.c_int, _p]),
    "cone_video_prepare_motion": (C.c_int, [_p, _p, _i64, _p, _p, _sz, C.c_int, _p]),
    "cone_video_prepare_motion_ex": (C.c_int, [_p, _p, _i32, _i64, _p, _p, _sz, C.c_int, _p]),
    "cone_adapter": (C.c_int, [_p, _p, _p, _i64, C.c_int, _p, _sz, C.c_int, _p]),
    "cone_linear": (C.c_int, [_p, _p, _p, _p, _i64, _i32, _i32, C.c_int, _p, _p, _p, _sz, C.c_int, _p]),
    "cone_encoder_tail": (C.c_int, [_p, _i32, _p, _p, _i64, _p, _i32, _p, _sz, _p]),
    "cone_frame_scores": (C.c_int, [_p, _i32, _p, _p, _i32, _i32, _i32, _p, _p, _p, C.c_int, _p]),
    "cone_window_ranklist": (C.c_int, [_p, _p, _p, _i32, _i32, _p, _p, _i32, _p]),
    "cone_prefilter_workspace_bytes": (_sz, [_p, _i64, _i32]),
    "cone_prefilter": (C.c_int, [_p, _p, _i64, _p, _i32, _i32, _p, _p, _p, _sz, _p]),
    "cone_prefilter_ex": (C.c_int, [_p, _p, _i32, _i64, _p, _i32, _i32, _i32, _p, _p, _p, _sz, _p]),
    "cone_ground_windows": (C.c_int, [_p, _p, _i64, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _i32, _i32, _i32,
                                      _p, _p, _p, _p, _p, _p, _sz, C.c_int, _p]),
    "cone_ground_windows_ex": (C.c_int, [_p, _p, _i32, _i64, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _i32, _i32, _i32,
                                         _p, _p, _p, _p, _p, _p, _sz, C.c_int, _p]),
    "cone_forward": (C.c_int, [_p, _p, _p, _p, _p, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _sz, C.c_int, _p]),
    "cone_clip_matching": (C.c_int, [_p, _p, _p, _p, _p, _i32, _i32, _i32, _p, _p, _sz, C.c_int, _p]),
    "cone_fuse_nms": (C.c_int, [_p, _p, _p, _p, _p, _i32, _i32, _i32, _f32, _f64, _i32, _i32, _p, _p, _p, _p, _p]),
    "cone_fuse_nms_ex": (C.c_int, [_p, _p, _p, _p, _p, _i32, _i32, _i32, _f32, _f64, _i32, _i32, _i32, _i32, _p, _p, _p, _p,
                                   _p]),
    "cone_fuse_nms_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "cone_fuse_nms_ws": (C.c_int, [_p, _p, _p, _p, _p, _i32, _i32, _i32, _f32, _f64, _i32, _i32, _i32, _i32, _p, _p, _p, _p,
                                   _p, _sz, _p]),
    "cone_temporal_nms": (C.c_int, [_p, _p, _p, _i32, _f64, _i32, _p, _p, _p]),
    "cone_eval_recall": (C.c_int, [_p, _p, _p, _i32, _i32, _p, _i32, _p, _i32, _i32, _p, _p, _p]),
    "cone_eval_window_recall": (C.c_int, [_p, _i32, _p, _i32, _f64, _i32, _p, _i32, _p, _p]),
    "cone_profile_enable": (None, [C.c_int]),
    "cone_profile_categories": (C.c_int, []),
    "cone_profile_name": (C.c_char_p, [C.c_int]),
    "cone_profile_read": (C.c_int, [_p, _p, _p, _p, C.c_int]),
    "cone_launch_count": (_i64, []),
    "cone_launch_count_reset": (None, []),
}


def load() -> C.CDLL:
    """Load (once) the CUDA library.  Raises ConeError if it has not been built."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise ConeError(f"{LIB_PATH} not found: build it with `python -m cone_b200.build` "
                            "(cone_b200 has no CPU or PyTorch fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the header and the library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().cone_last_error().decode("utf-8", "replace")
        raise ConeError(f"{what or 'cone_b200'} failed (code {rc}): {msg}")


def launch_count() -> int:
    return int(load().cone_launch_count())


def reset_launch_count() -> None:
    load().cone_launch_count_reset()
