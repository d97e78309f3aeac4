"""ctypes binding of the C ABI in include/dvfe.h (libdvfe.so, built in-tree by __graft_entry__.build()).

There is no Python or CPU fallback: if the shared library is missing, or no CUDA device is visible
when a compute entry point is called, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DVFE_LIB", os.path.join(_HERE, "libdvfe.so"))   # DVFE_LIB: development override

DVFE_OK = 0
ERRORS = {-1: "DVFE_ERR_INVALID", -2: "DVFE_ERR_CUDA", -3: "DVFE_ERR_CONFIG", -4: "DVFE_ERR_CAPACITY",
          -5: "DVFE_ERR_NO_DEVICE"}


class DvfeError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERRORS.get(code, code)}: {msg}")
        self.code = code


class Camera(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("fx", "fy", "cx", "cy", "k1", "k2", "p1", "p2")]


class Config(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("width", "height", "n_streams", "stereo", "max_cnt", "min_dist",
                                       "max_dynamic_cnt", "min_dynamic_dist", "flow_back", "use_mask_morphology",
                                       "mask_morphology_size", "lk_max_level", "max_instances", "device")] + \
               [("cam0", Camera), ("cam1", Camera), ("n_groups", C.c_int), ("reserved", C.c_int)]


class Obs(C.Structure):
    _fields_ = [("id", C.c_uint32), ("cam", C.c_int32), ("v", C.c_double * 7)]


OBS_DTYPE = np.dtype([("id", np.uint32), ("cam", np.int32), ("v", np.float64, (7,))])


class InstObs(C.Structure):
    _fields_ = [("inst_id", C.c_uint32), ("id", C.c_uint32), ("is_stereo", C.c_int32), ("reserved", C.c_int32),
                ("point", C.c_double * 3), ("vel", C.c_double * 2), ("point_right", C.c_double * 3),
                ("vel_right", C.c_double * 2), ("uv", C.c_double * 2), ("disp", C.c_double)]


INST_OBS_DTYPE = np.dtype([("inst_id", np.uint32), ("id", np.uint32), ("is_stereo", np.int32), ("reserved", np.int32),
                           ("point", np.float64, (3,)), ("vel", np.float64, (2,)),
                           ("point_right", np.float64, (3,)), ("vel_right", np.float64, (2,)),
                           ("uv", np.float64, (2,)), ("disp", np.float64)])


class InstIn(C.Structure):
    _fields_ = [("track_id", C.c_uint32), ("x", C.c_int32), ("y", C.c_int32), ("w", C.c_int32), ("h", C.c_int32),
                ("mask", C.c_void_p), ("mask_pitch", C.c_int32), ("disp", C.c_void_p), ("disp_pitch", C.c_int32), ("label_bit", C.c_int32)]


class InstInfo(C.Structure):
    _fields_ = [("track_id", C.c_uint32), ("lost_num", C.c_int32), ("is_curr_visible", C.c_int32), ("has_box", C.c_int32),
                ("x", C.c_int32), ("y", C.c_int32), ("w", C.c_int32), ("h", C.c_int32)]


class FrameDesc(C.Structure):
    """dvfe_frame: one camera's images of a step (dvfe_track_frames)"""
    _fields_ = [("left", C.c_void_p), ("right", C.c_void_p), ("mask", C.c_void_p), ("pitch", C.c_int32), ("mask_pitch", C.c_int32),
                ("exist_inst", C.c_int32), ("flags", C.c_uint32), ("time0", C.c_double)]


class State(C.Structure):
    _fields_ = [("n", C.c_int), ("next_id", C.c_uint32), ("prev_time", C.c_double),
                ("ids", C.c_void_p), ("track_cnt", C.c_void_p), ("last_points", C.c_void_p),
                ("prev_un", C.c_void_p), ("right_prev_un", C.c_void_p), ("right_prev_valid", C.c_void_p)]


# every symbol include/dvfe.h declares (checked by tests/test_abi.py)
SYMBOLS = [
    "dvfe_create", "dvfe_destroy", "dvfe_config_from_yaml", "dvfe_last_error", "dvfe_version",
    "dvfe_kernel_launches", "dvfe_set_stream", "dvfe_profile", "dvfe_profile_read", "dvfe_track_image", "dvfe_track_image_async", "dvfe_wait", "dvfe_track_image_device_async", "dvfe_set_lk_mode", "dvfe_set_lk_mode_site", "dvfe_track_image_device", "dvfe_track_semantic_image",
    "dvfe_insts_track", "dvfe_insts_track_batch", "dvfe_get_features", "dvfe_insts_output", "dvfe_get_state", "dvfe_set_state",
    "dvfe_op_build_pyramid", "dvfe_op_lk", "dvfe_op_min_eigen_val", "dvfe_op_good_features",
    "dvfe_op_disc_mask", "dvfe_op_erode_rect", "dvfe_op_lift_projective", "dvfe_op_bgr_to_gray", "dvfe_op_merge_masks",
    "dvfe_op_remap", "dvfe_set_input", "dvfe_set_undistort_maps", "dvfe_track_dynamic_async", "dvfe_op_punch_out", "dvfe_insts_table", "dvfe_track_dynamic_ex",
    "dvfe_op_reject_with_f", "dvfe_op_detect_extra_points", "dvfe_op_build_pyramid_bordered", "dvfe_set_detect_mode", "dvfe_op_good_features_cuda",
    "dvfe_track_image_ex", "dvfe_track_semantic_ex", "dvfe_track_dynamic_ex2",
    "dvfe_set_stream_camera", "dvfe_set_stream_undistort_maps", "dvfe_camera_from_yaml",
    "dvfe_export_stream", "dvfe_import_stream",
    "dvfe_track_frames", "dvfe_track_semantic_frames", "dvfe_track_dynamic_frames",
]
# every symbol include/dvfe/reject_with_f.h declares (the companion header of the in-step RejectWithF)
REJECT_SYMBOLS = ["dvfe_set_reject_with_f", "dvfe_f_threshold_from_yaml"]

# dvfe_track_image_ex / _semantic_ex / _dynamic_ex2: per-stream frame flags; dvfe_track_image_ex's step flags (include/dvfe.h)
FRAME_SKIP, FRAME_NO_RIGHT, FRAME_RESET = 1, 2, 4
STEP_DEVICE_INPUT = 1

_lib = None


def lib() -> C.CDLL:
    """Load libdvfe.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              f"(dynamic_vins_b200 has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.dvfe_last_error.restype = C.c_char_p
        L.dvfe_last_error.argtypes = [C.c_void_p]
        L.dvfe_version.restype = C.c_char_p
        L.dvfe_kernel_launches.restype = C.c_ulonglong
        L.dvfe_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
        L.dvfe_destroy.argtypes = [C.c_void_p]
        L.dvfe_destroy.restype = None
        L.dvfe_config_from_yaml.argtypes = [C.c_char_p, C.POINTER(Config)]
        L.dvfe_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        L.dvfe_profile.argtypes = [C.c_void_p, C.c_int]
        L.dvfe_profile_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_long)]
        L.dvfe_track_image.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
        L.dvfe_track_image_async.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
        L.dvfe_wait.argtypes = [C.c_void_p]
        L.dvfe_track_image_device_async.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
        L.dvfe_track_image_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p, C.c_uint]
        L.dvfe_set_lk_mode.argtypes = [C.c_void_p, C.c_int, C.c_double]
        L.dvfe_set_lk_mode_site.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double]
        L.dvfe_track_image_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
        L.dvfe_track_semantic_image.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int,
                                                C.c_void_p, C.c_void_p]
        L.dvfe_insts_track.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_double]
        L.dvfe_insts_track_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.dvfe_get_features.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.dvfe_insts_output.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.dvfe_get_state.argtypes = [C.c_void_p, C.c_int, C.POINTER(State), C.c_int]
        L.dvfe_set_state.argtypes = [C.c_void_p, C.c_int, C.POINTER(State)]
        L.dvfe_op_build_pyramid.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.POINTER(C.c_int)]
        L.dvfe_op_lk.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                 C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.dvfe_op_min_eigen_val.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.dvfe_op_good_features_cuda.argtypes = L.dvfe_op_good_features.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                            C.c_int, C.c_double, C.c_double, C.c_void_p, C.POINTER(C.c_int),
                                            C.POINTER(C.c_int)]
        L.dvfe_op_disc_mask.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int]
        L.dvfe_op_erode_rect.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.dvfe_op_lift_projective.argtypes = [C.POINTER(Camera), C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_void_p]
        L.dvfe_op_bgr_to_gray.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.dvfe_op_remap.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.dvfe_track_dynamic_async.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_void_p]
        L.dvfe_op_punch_out.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.dvfe_track_dynamic_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint]
        L.dvfe_track_dynamic_ex2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint]
        L.dvfe_track_semantic_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_uint]
        L.dvfe_insts_table.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.dvfe_set_input.argtypes = [C.c_void_p, C.c_int]
        L.dvfe_set_undistort_maps.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.dvfe_set_stream_camera.argtypes = [C.c_void_p, C.c_int, C.POINTER(Camera), C.POINTER(Camera)]
        L.dvfe_set_stream_undistort_maps.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.dvfe_camera_from_yaml.argtypes = [C.c_char_p, C.POINTER(Camera)]
        L.dvfe_export_stream.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.dvfe_import_stream.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_size_t]
        L.dvfe_track_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_uint]
        L.dvfe_track_semantic_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_uint]
        L.dvfe_track_dynamic_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint]
        L.dvfe_op_merge_masks.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.dvfe_set_detect_mode.argtypes = [C.c_void_p, C.c_int]
        L.dvfe_set_reject_with_f.argtypes = [C.c_void_p, C.c_double]
        L.dvfe_f_threshold_from_yaml.argtypes = [C.c_char_p, C.POINTER(C.c_double)]
        L.dvfe_op_build_pyramid_bordered.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.dvfe_op_reject_with_f.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p,
                                            C.POINTER(C.c_int)]
        L.dvfe_op_detect_extra_points.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                                  C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != DVFE_OK:
        raise DvfeError(rc, lib().dvfe_last_error(None).decode("utf-8", "replace"))


def ptr(a) -> C.c_void_p:
    return None if a is None else C.c_void_p(a.ctypes.data)
