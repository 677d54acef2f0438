"""ctypes binding of csrc/libagt.so (the C ABI declared in include/agt.h).

There is deliberately no fallback: if the shared library is missing or no B200
is visible, every compute entry point raises.  Error codes map to the exception
types the reference raises at the same places (SURVEY.md 8b): AGT_ERR_INVALID ->
ValueError, AGT_ERR_NOT_READY / AGT_ERR_CUDA / AGT_ERR_NO_DEVICE -> RuntimeError.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

LIB_PATH = Path(__file__).resolve().parent / "csrc" / "libagt.so"

AGT_MAX_LEVELS = 4
AGT_MAX_TAGS = 16
AGT_MAX_POINTS = 64
AGT_STREAM_STATE_DOUBLES = 64
AGT_OK, AGT_ERR_INVALID, AGT_ERR_CUDA, AGT_ERR_NOT_READY, AGT_ERR_NO_DEVICE = 0, -1, -2, -3, -4
DPR_NONE, DPR_CONVERGED, DPR_MAX_EVALS, DPR_LAMBDA = 0, 1, 2, 3


class AgtPyramid(C.Structure):
    _fields_ = [("levels", C.c_int32),
                ("width", C.c_int32 * AGT_MAX_LEVELS),
                ("height", C.c_int32 * AGT_MAX_LEVELS),
                ("pitch", C.c_int64 * AGT_MAX_LEVELS),
                ("frame_stride", C.c_int64 * AGT_MAX_LEVELS),
                ("data", C.c_void_p * AGT_MAX_LEVELS)]


class AgtLibraryError(RuntimeError):
    pass


_lib = None

_VP, _I, _I64, _D = C.c_void_p, C.c_int, C.c_int64, C.c_double
_PYR = C.POINTER(AgtPyramid)

# name -> (restype, argtypes); every symbol include/agt.h declares
PROTOTYPES = {
    "agt_version": (_I, []),
    "agt_device_count": (_I, []),
    "agt_create": (_I, [_I, C.POINTER(_VP)]),
    "agt_destroy": (_I, [_VP]),
    "agt_last_error": (C.c_char_p, [_VP]),
    "agt_set_stream": (_I, [_VP, _VP]),
    "agt_sync": (_I, [_VP]),
    "agt_launch_count": (_I64, [_VP]),
    "agt_set_camera": (_I, [_VP, C.POINTER(_D), C.POINTER(_D), _I]),
    "agt_set_model": (_I, [_VP, _VP, _VP, _I, _VP, _VP, _I, _D]),
    "agt_bgr_to_gray": (_I, [_VP, _VP, _I, _I, _I64, _I64, _VP, _I64, _I64, _I]),
    "agt_set_undistort": (_I, [_VP, C.POINTER(_D), _I, _I, _I, _I, _I, _I]),
    "agt_undistort_to_gray": (_I, [_VP, _VP, _I, _I, _I, _I64, _I64, _VP, _I64, _I64, _I]),
    "agt_undistort_to_gray_host": (_I, [_VP, _VP, _I, _I, _I, _VP]),
    "agt_set_tag_family": (_I, [_VP, _VP, _I]),
    "agt_set_tag_threshold": (_I, [_VP, _I]),
    "agt_decode_tags": (_I, [_VP, _VP, _I, _I, _I64, _I64, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I, _I]),
    "agt_detect_tags": (_I, [_VP, _VP, _I, _I, _I64, _I64, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP]),
    "agt_detect_tags_host": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP]),
    "agt_detect_tags_roi": (_I, [_VP, _VP, _I, _I, _I64, _I64, _I, _VP, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP]),
    "agt_tag_quads": (_I, [_VP, _VP, _I, _I, _I64, _I64, _I, _VP, _I, _I, _I, _VP, _VP, _VP, _VP, _VP]),
    "agt_track_rects": (_I, [_VP, _VP, _D, _I, _I, _I, _VP, _I]),
    "agt_pack_detections": (_I, [_VP, _VP, _VP, _VP, _VP, _I, _VP, _I, C.c_float, _VP, _VP, _VP, _VP, _I]),
    "agt_draw_points": (_I, [_VP, _VP, _I, _I, _I64, _I64, _VP, _VP, _I, _I, _I, _I, _I, _I, _I, _I]),
    "agt_corner_subpix": (_I, [_VP, _VP, _I, _I, _I64, _I64, _VP, _VP, _VP, _I, _I, _I, _I, _D]),
    "agt_corner_subpix_host": (_I, [_VP, _VP, _I, _I, _VP, _I, _I, _I, _D]),
    "agt_bgr_to_gray_host": (_I, [_VP, _VP, _I, _I, _VP]),
    "agt_undistort_frames": (_I, [_VP, _VP, _I, _I, _I, _I64, _I64, _VP, _I64, _I64, _I]),
    "agt_undistort_frame_host": (_I, [_VP, _VP, _I, _I, _I, _VP, _VP]),
    "agt_pyr_down": (_I, [_VP, _VP, _I, _I, _I64, _I64, _VP, _I64, _I64, _I]),
    "agt_build_pyramid": (_I, [_VP, _PYR, _I]),
    "agt_build_pyramid_roi": (_I, [_VP, _PYR, _VP, _I, _I]),
    "agt_build_pyramid_masked": (_I, [_VP, _PYR, _VP, _I, _I]),
    "agt_dpr_rects": (_I, [_VP, _PYR, _VP, _I, _VP, _I]),
    "agt_any_flag": (_I, [_VP, _VP, _I, _VP, _I]),
    "agt_scharr": (_I, [_VP, _VP, _I, _I, _I64, _I64, _VP, _I]),
    "agt_lk": (_I, [_VP, _PYR, _PYR, _VP, _VP, _VP, _VP, _I, _I]),
    "agt_lk_fallback": (_I, [_VP, _PYR, _PYR, _VP, _VP, _VP, _VP, _VP, _I, _I]),
    "agt_lk_rects": (_I, [_VP, _PYR, _VP, _VP, _I, _I, _VP, _I, _I]),
    "agt_lk_roi": (_I, [_VP, _PYR, _PYR, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _VP, _VP, _I, _I]),
    "agt_pnp": (_I, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I]),
    "agt_streams_front": (_I, [_VP] * 11 + [_I] + [_VP] * 6 + [_I, _I]),
    "agt_project": (_I, [_VP, _VP, _VP, _VP, _I, _I]),
    "agt_ape_prepare": (_I, [_VP, _VP, _VP, _VP, _I, _I]),
    "agt_ape_update": (_I, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I]),
    "agt_accept_gate": (_I, [_VP, _VP, _VP, _VP, _VP, _I]),
    "agt_ape_commit": (_I, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _VP, _VP, _VP, _I, _I]),
    "agt_refine": (_I, [_VP, _PYR, _VP, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I]),
    "agt_refine_fused": (_I, [_VP, _PYR, _VP, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I]),
    "agt_lk_merge": (_I, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I]),
    "agt_select_best": (_I, [_VP, _VP, _VP, _VP, _I, _VP, _VP, _I]),
    "agt_render": (_I, [_VP, _VP, _VP, _VP, _I, _I, _I64, _I64, _VP, _VP, _I, _D, _D, _I, _I]),
    "agt_solve_pnp_host": (_I, [_VP, _VP, _VP, _I, _I, _VP, C.POINTER(_I), C.POINTER(C.c_float)]),
    "agt_project_host": (_I, [_VP, _VP, _I, _VP, _VP]),
    "agt_lk_host": (_I, [_VP, _VP, _VP, _I, _I, _I, _VP, _I, _VP, _VP, _VP]),
    "agt_pyramid_host": (_I, [_VP, _VP, _I, _I, _I, C.POINTER(_VP)]),
    "agt_scharr_host": (_I, [_VP, _VP, _I, _I, _VP]),
    "agt_set_roi_upload": (_I, [_VP, _I]),
    "agt_set_upload_threads": (_I, [_VP, _I]),
    "agt_last_h2d_bytes": (_I64, [_VP]),
    "agt_refine_host": (_I, [_VP, _VP, _I, _I, _I, _I, _VP, _I, _VP, _VP, _VP, _VP, _VP, _VP]),
    "agt_pose_covariance": (_I, [_VP, _PYR, _VP, _VP, _I, _VP, _VP, _VP, _VP, _VP, _VP, _I]),
    "agt_pose_covariance_host": (_I, [_VP, _VP, _I, _I, _I, _I, _VP, _VP, _I, _VP, _VP, _VP, _VP, _VP]),
}


def load() -> C.CDLL:
    """Load libagt.so and attach prototypes.  Raises AgtLibraryError if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise AgtLibraryError(
            f"{LIB_PATH} is missing: build it with `python -m accurate_aprilgroup_tracking_b200._build` "
            "(nvcc, sm_100a).  There is no CPU fallback for the tracking path.")
    try:
        lib = C.CDLL(str(LIB_PATH))
    except OSError as exc:
        raise AgtLibraryError(f"cannot load {LIB_PATH}: {exc}") from exc
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(ctx_handle, rc: int, what: str = "") -> None:
    if rc == AGT_OK:
        return
    lib = load()
    msg = lib.agt_last_error(ctx_handle)
    text = (msg.decode("utf-8", "replace") if msg else "") or what
    if rc == AGT_ERR_INVALID:
        raise ValueError(text)
    raise RuntimeError(f"libagt error {rc}: {text}")
