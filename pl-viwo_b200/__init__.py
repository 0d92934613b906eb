"""plviwo_b200 — Python binding (ctypes) of the B200-native PL-VIWO visual front end.

The product is ``libplviwo_fe.so`` (hand-written sm_100a kernels + C++ host trackers behind the C ABI in
``include/plviwo_fe.h``).  This module only marshals NumPy arrays across that ABI for tests and benchmarks and
mirrors the reference's tracker interface (``feed_new_camera``, ``get_last_obs``, ``get_last_ids``,
``get_feature_database`` — ov_core/src/track/TrackBase.h:72-196, PL-VIWO/src/update/cam/TrackLSD.h:84-99).
There is no CPU implementation behind it: if the library is missing or no GPU is present every compute call
raises ``FrontEndError``.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # one hardware queue per stream (see INTEGRATION.md)
_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libplviwo_fe.so")

FE_OK, FE_BAD_ARG, FE_NO_DEVICE, FE_CUDA_ERROR, FE_OVERFLOW, FE_INTERNAL = range(6)
HIST_NONE, HIST_HISTOGRAM, HIST_CLAHE = 0, 1, 2
# camera models (FeCameraModel): ov_core's CamRadtan and CamEqui, fixed when a front end is created
CAM_RADTAN, CAM_EQUI = 0, 1
FE_CAM_RADTAN, FE_CAM_EQUI = CAM_RADTAN, CAM_EQUI
_STATUS = {0: "FE_OK", 1: "FE_BAD_ARG", 2: "FE_NO_DEVICE", 3: "FE_CUDA_ERROR", 4: "FE_OVERFLOW", 5: "FE_INTERNAL"}
HOST_STAGES = ["submit", "detection", "matching", "ransac", "lines", "collect", "line_wait", "predet_wait",
               "speculate", "assemble", "line_assign", "spec_launch", "lk_launch", "lk_wait", "line_match", "line_rows"]
STAGES = ["h2d", "hist", "eq_pyr1", "pyr_rest", "fast", "subpix", "lk", "canny", "fld", "fld_ccl", "fld_walk", "fld_seg",
          "line_frames"]   # line_frames: launches[] only (frames carried by the timed line-path launches)
TAP_PYR_LEVEL0, TAP_HALF, TAP_EDGES, TAP_FAST_LAST, TAP_LK_LAST, TAP_SUBPIX_LAST, TAP_FLD_LAST = 0, 32, 33, 34, 35, 36, 37


class FrontEndError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("%s: %s" % (_STATUS.get(code, code), msg))
        self.code = code


class FeConfig(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("num_features", C.c_int32), ("fast_threshold", C.c_int32),
        ("grid_x", C.c_int32), ("grid_y", C.c_int32), ("min_px_dist", C.c_int32), ("pyr_levels", C.c_int32),
        ("win_size", C.c_int32), ("histogram_method", C.c_int32), ("numaruco", C.c_int32), ("use_lines", C.c_int32),
        ("fld_length_threshold", C.c_int32), ("fld_distance_threshold", C.c_float), ("canny_th1", C.c_float),
        ("canny_th2", C.c_float), ("line_min_length", C.c_float), ("line_samples", C.c_int32), ("lookahead", C.c_int32), ("downsample", C.c_int32),
        ("K", C.c_double * 4), ("D", C.c_double * 4),
    ]


class FePointRow(C.Structure):
    _fields_ = [("id", C.c_uint64), ("u", C.c_float), ("v", C.c_float), ("un", C.c_float), ("vn", C.c_float)]


class FeLineRow(C.Structure):
    _fields_ = [("id", C.c_uint64), ("line", C.c_float * 4), ("line_n", C.c_float * 4), ("D", C.c_int32),
                ("n_pts", C.c_int32), ("pt_offset", C.c_int32), ("matched", C.c_int32)]


class FeLinePoint(C.Structure):
    _fields_ = [("pid", C.c_int32), ("dist", C.c_float), ("u", C.c_float), ("v", C.c_float)]


class FeFrameInfo(C.Structure):
    _fields_ = [("timestamp", C.c_double), ("n_point_rows", C.c_int32), ("n_line_rows", C.c_int32),
                ("n_last_obs", C.c_int32), ("reset", C.c_int32), ("first_frame", C.c_int32), ("n_detected", C.c_int32),
                ("n_lk_in", C.c_int32), ("n_klt_ok", C.c_int32), ("n_ransac_ok", C.c_int32),
                ("n_lines_detected", C.c_int32), ("n_line_matches", C.c_int32), ("detection_ran", C.c_int32),
                ("reserved", C.c_int32)]


class FeStereoInfo(C.Structure):
    _fields_ = [("timestamp", C.c_double), ("n_point_rows", C.c_int32 * 2), ("n_last_obs", C.c_int32 * 2), ("reset", C.c_int32),
                ("first_frame", C.c_int32), ("detection_ran", C.c_int32 * 2), ("n_detected", C.c_int32 * 2),
                ("n_stereo_new", C.c_int32), ("n_lk_in", C.c_int32 * 2), ("n_klt_ok", C.c_int32 * 2),
                ("n_ransac_ok", C.c_int32 * 2), ("n_stereo_rows", C.c_int32), ("n_line_rows", C.c_int32),
                ("n_lines_detected", C.c_int32), ("n_line_matches", C.c_int32)]


class FePlayStats(C.Structure):
    _fields_ = [("frames", C.c_uint64), ("point_rows", C.c_uint64), ("line_rows", C.c_uint64), ("resets", C.c_uint64),
                ("checksum", C.c_double)]


class FeStageTimes(C.Structure):
    _fields_ = [("ms", C.c_double * 16), ("launches", C.c_uint64 * 16), ("frames", C.c_uint64),
                ("kernel_launches_total", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("host_ms", C.c_double * 16)]


GROUP_KERNELS = ["hist", "eq_pyr1", "pyr_rest", "fast", "select", "subpix", "canny", "ccl", "walk", "segments", "detect", "lk", "gate",
                 "lines", "accept", "cands"]


class FeGroupTimes(C.Structure):
    _fields_ = [("ms", C.c_double * 16), ("launches", C.c_uint64 * 16), ("frames", C.c_uint64 * 16), ("ticks", C.c_uint64),
                ("frames_total", C.c_uint64), ("kernel_launches_total", C.c_uint64), ("h2d_bytes", C.c_uint64),
                ("d2h_bytes", C.c_uint64), ("fast_cells", C.c_uint64)]


POINT_ROW_DTYPE = np.dtype([("id", "<u8"), ("u", "<f4"), ("v", "<f4"), ("un", "<f4"), ("vn", "<f4")])
LINE_ROW_DTYPE = np.dtype([("id", "<u8"), ("line", "<f4", (4,)), ("line_n", "<f4", (4,)), ("D", "<i4"), ("n_pts", "<i4"),
                           ("pt_offset", "<i4"), ("matched", "<i4")])
LINE_POINT_DTYPE = np.dtype([("pid", "<i4"), ("dist", "<f4"), ("u", "<f4"), ("v", "<f4")])

_lib = None

# every symbol include/plviwo_fe.h declares (tests/test_abi.py checks the header against this list and the .so)
EXPORTS = [
    "plviwo_fe_abi_version", "plviwo_fe_default_config", "plviwo_fe_device_count", "plviwo_fe_create", "plviwo_fe_destroy",
    "plviwo_fe_last_error", "plviwo_fe_classify_lines", "plviwo_fe_set_calib", "plviwo_fe_set_num_features", "plviwo_fe_change_feat_id", "plviwo_fe_feed",
    "plviwo_fe_feed_device", "plviwo_fe_submit", "plviwo_fe_collect", "plviwo_fe_play", "plviwo_fe_get_point_rows", "plviwo_fe_get_last_obs",
    "plviwo_fe_get_line_rows", "plviwo_fe_get_line_points", "plviwo_fe_get_line_samples", "plviwo_fe_get_state",
    "plviwo_fe_set_state", "plviwo_fe_enable_taps", "plviwo_fe_tap", "plviwo_fe_enable_timing", "plviwo_fe_get_stage_times",
    "plviwo_op_equalize_pyramid", "plviwo_op_clahe", "plviwo_op_fast_cell", "plviwo_op_sort_corners", "plviwo_op_corner_subpix", "plviwo_op_lk", "plviwo_op_lk_warp", "plviwo_op_undistort",
    "plviwo_op_canny_half", "plviwo_op_ccl_tiles", "plviwo_op_fld", "plviwo_op_image_kernels_time", "plviwo_op_ransac_fundamental",
    "plviwo_fe_stereo_create", "plviwo_fe_stereo_destroy", "plviwo_fe_stereo_last_error", "plviwo_fe_stereo_set_calib",
    "plviwo_fe_stereo_set_num_features", "plviwo_fe_stereo_change_feat_id", "plviwo_fe_stereo_feed", "plviwo_fe_stereo_submit",
    "plviwo_fe_stereo_collect", "plviwo_fe_stereo_get_point_rows", "plviwo_fe_stereo_get_last_obs", "plviwo_fe_stereo_get_state",
    "plviwo_fe_stereo_set_state", "plviwo_fe_stereo_get_stage_times", "plviwo_fe_stereo_get_line_rows",
    "plviwo_fe_stereo_get_line_points", "plviwo_fe_stereo_classify_lines", "plviwo_op_line_match",
    "plviwo_op_assign_points",
    "plviwo_fe_group_create", "plviwo_fe_group_destroy", "plviwo_fe_group_last_error", "plviwo_fe_group_set_calib", "plviwo_fe_group_set_camera",
    "plviwo_fe_group_submit", "plviwo_fe_group_collect", "plviwo_fe_group_play", "plviwo_fe_group_get_point_rows",
    "plviwo_fe_group_get_last_obs", "plviwo_fe_group_get_line_rows", "plviwo_fe_group_get_line_points",
    "plviwo_fe_group_get_line_samples",
    "plviwo_fe_group_get_state", "plviwo_fe_group_set_state", "plviwo_fe_group_tap", "plviwo_fe_group_enable_timing",
    "plviwo_fe_group_get_times", "plviwo_fe_set_camera", "plviwo_fe_get_currid", "plviwo_fe_set_currid",
    "plviwo_fe_stereo_set_camera",
    "plviwo_fe_stereo_group_create", "plviwo_fe_stereo_group_destroy", "plviwo_fe_stereo_group_last_error", "plviwo_fe_stereo_group_set_calib", "plviwo_fe_stereo_group_set_camera", "plviwo_fe_stereo_group_submit",
    "plviwo_fe_create_model", "plviwo_fe_stereo_create_model", "plviwo_fe_group_create_model", "plviwo_fe_stereo_group_create_model",
    "plviwo_op_undistort_equi",
    "plviwo_fe_stereo_group_collect", "plviwo_fe_stereo_group_play", "plviwo_fe_stereo_group_get_point_rows", "plviwo_fe_stereo_group_get_last_obs", "plviwo_fe_stereo_group_get_line_rows", "plviwo_fe_stereo_group_get_line_points", "plviwo_fe_stereo_group_get_state", "plviwo_fe_stereo_group_set_state",
]


def lib() -> C.CDLL:
    """Loads libplviwo_fe.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FrontEndError(FE_INTERNAL, "%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                             "(there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.plviwo_fe_last_error.restype = C.c_char_p
        L.plviwo_fe_last_error.argtypes = [C.c_void_p]
        L.plviwo_fe_create.argtypes = [C.POINTER(FeConfig), C.c_int, C.POINTER(C.c_void_p)]
        L.plviwo_fe_create_model.argtypes = [C.POINTER(FeConfig), C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.plviwo_fe_stereo_create_model.argtypes = [C.POINTER(FeConfig), C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                                    C.c_int, C.POINTER(C.c_void_p)]
        L.plviwo_fe_group_create_model.argtypes = [C.POINTER(FeConfig), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.plviwo_fe_stereo_group_create_model.argtypes = [C.POINTER(FeConfig), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.plviwo_op_undistort_equi.argtypes = [C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                               C.c_void_p]
        L.plviwo_fe_destroy.argtypes = [C.c_void_p]
        L.plviwo_fe_set_calib.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.plviwo_fe_set_camera.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.plviwo_fe_get_currid.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        L.plviwo_fe_set_currid.argtypes = [C.c_void_p, C.c_uint64]
        L.plviwo_fe_stereo_set_camera.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.plviwo_fe_set_num_features.argtypes = [C.c_void_p, C.c_int]
        L.plviwo_fe_classify_lines.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.plviwo_fe_change_feat_id.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64]
        L.plviwo_fe_feed.argtypes = [C.c_void_p, C.c_double, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                     C.c_void_p, C.POINTER(FeFrameInfo)]
        L.plviwo_fe_feed_device.argtypes = L.plviwo_fe_feed.argtypes
        L.plviwo_fe_submit.argtypes = [C.c_void_p, C.c_double, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
        L.plviwo_fe_collect.argtypes = [C.c_void_p, C.POINTER(FeFrameInfo)]
        L.plviwo_fe_play.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.POINTER(C.c_double),
                                     C.POINTER(C.c_double), C.POINTER(FePlayStats)]
        for name in ("plviwo_fe_get_point_rows", "plviwo_fe_get_line_rows", "plviwo_fe_get_line_points"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_fe_get_last_obs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_fe_get_line_samples.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_fe_get_state.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.plviwo_fe_set_state.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.plviwo_fe_tap.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.plviwo_fe_enable_timing.argtypes = [C.c_void_p, C.c_int]
        L.plviwo_fe_enable_taps.argtypes = [C.c_void_p, C.c_int]
        L.plviwo_fe_get_stage_times.argtypes = [C.c_void_p, C.POINTER(FeStageTimes), C.c_int]
        L.plviwo_fe_stereo_last_error.restype = C.c_char_p
        L.plviwo_fe_stereo_last_error.argtypes = [C.c_void_p]
        L.plviwo_fe_stereo_create.argtypes = [C.POINTER(FeConfig), C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int,
                                              C.POINTER(C.c_void_p)]
        L.plviwo_fe_stereo_destroy.argtypes = [C.c_void_p]
        L.plviwo_fe_stereo_set_calib.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.plviwo_fe_stereo_set_num_features.argtypes = [C.c_void_p, C.c_int]
        L.plviwo_fe_stereo_change_feat_id.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64]
        L.plviwo_fe_stereo_feed.argtypes = [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                            C.c_void_p, C.c_int, C.c_void_p, C.POINTER(FeStereoInfo)]
        L.plviwo_fe_stereo_submit.argtypes = [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                              C.c_void_p, C.c_int, C.c_void_p]
        L.plviwo_fe_stereo_get_line_rows.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_fe_stereo_get_line_points.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_fe_stereo_classify_lines.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.plviwo_fe_stereo_collect.argtypes = [C.c_void_p, C.POINTER(FeStereoInfo)]
        L.plviwo_fe_stereo_get_point_rows.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_fe_stereo_get_last_obs.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_fe_stereo_get_state.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.plviwo_fe_stereo_set_state.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.plviwo_fe_stereo_get_stage_times.argtypes = [C.c_void_p, C.POINTER(FeStageTimes), C.c_int]
        L.plviwo_fe_default_config.argtypes = [C.POINTER(FeConfig)]
        L.plviwo_fe_default_config.restype = None
        L.plviwo_fe_device_count.argtypes = [C.POINTER(C.c_int)]
        L.plviwo_op_equalize_pyramid.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.plviwo_op_clahe.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.plviwo_op_fast_cell.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_op_corner_subpix.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
        L.plviwo_op_sort_corners.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]
        L.plviwo_op_lk.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_int]
        L.plviwo_op_lk_warp.argtypes = L.plviwo_op_lk.argtypes
        L.plviwo_op_undistort.argtypes = [C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p]
        L.plviwo_op_canny_half.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p]
        L.plviwo_op_ccl_tiles.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_int, C.POINTER(C.c_int)]
        L.plviwo_op_fld.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_int,
                                    C.POINTER(C.c_int)]
        L.plviwo_op_image_kernels_time.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]
        L.plviwo_op_ransac_fundamental.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_void_p,
                                                   C.POINTER(C.c_int)]
        L.plviwo_fe_group_last_error.restype = C.c_char_p
        L.plviwo_fe_group_last_error.argtypes = [C.c_void_p]
        L.plviwo_fe_group_create.argtypes = [C.POINTER(FeConfig), C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.plviwo_fe_group_destroy.argtypes = [C.c_void_p]
        L.plviwo_fe_group_set_calib.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.plviwo_fe_group_set_camera.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.plviwo_fe_group_submit.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_void_p), C.c_int, C.c_int,
                                             C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_double)]
        L.plviwo_fe_group_collect.argtypes = [C.c_void_p, C.POINTER(FeFrameInfo)]
        L.plviwo_fe_group_play.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.POINTER(C.c_double),
                                           C.POINTER(C.c_double), C.POINTER(FePlayStats)]
        for name in ("plviwo_fe_group_get_point_rows", "plviwo_fe_group_get_line_rows", "plviwo_fe_group_get_line_points"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_fe_group_get_last_obs.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_fe_group_get_line_samples.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_fe_group_get_state.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.plviwo_fe_group_set_state.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
        L.plviwo_fe_group_tap.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.plviwo_fe_group_enable_timing.argtypes = [C.c_void_p, C.c_int]
        L.plviwo_fe_group_get_times.argtypes = [C.c_void_p, C.POINTER(FeGroupTimes), C.c_int]
        L.plviwo_fe_stereo_group_last_error.restype = C.c_char_p
        L.plviwo_fe_stereo_group_last_error.argtypes = [C.c_void_p]
        L.plviwo_fe_stereo_group_create.argtypes = [C.POINTER(FeConfig), C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.plviwo_fe_stereo_group_destroy.argtypes = [C.c_void_p]
        L.plviwo_fe_stereo_group_set_calib.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.plviwo_fe_stereo_group_set_camera.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double),
                                                        C.POINTER(C.c_double)]
        L.plviwo_fe_stereo_group_submit.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                                    C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int,
                                                    C.POINTER(C.c_double)]
        L.plviwo_fe_stereo_group_collect.argtypes = [C.c_void_p, C.POINTER(FeStereoInfo)]
        L.plviwo_fe_stereo_group_play.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_int, C.c_int,
                                                  C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(FePlayStats)]
        L.plviwo_fe_stereo_group_get_point_rows.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_fe_stereo_group_get_last_obs.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                                          C.POINTER(C.c_int)]
        for name in ("plviwo_fe_stereo_group_get_line_rows", "plviwo_fe_stereo_group_get_line_points"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.plviwo_fe_stereo_group_get_state.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.plviwo_fe_stereo_group_set_state.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
        _lib = L
    return _lib


def _check(rc: int, handle=None):
    if rc != FE_OK:
        msg = lib().plviwo_fe_last_error(handle)
        raise FrontEndError(rc, msg.decode() if msg else "")


def default_config(**kw) -> FeConfig:
    cfg = FeConfig()
    lib().plviwo_fe_default_config(C.byref(cfg))
    for k, v in kw.items():
        if k in ("K", "D"):
            for i in range(4):
                getattr(cfg, k)[i] = float(v[i])
        else:
            if not hasattr(cfg, k):
                raise AttributeError(k)
            setattr(cfg, k, v)
    return cfg


def device_count() -> int:
    n = C.c_int(0)
    lib().plviwo_fe_device_count(C.byref(n))
    return n.value


# ------------------------------------------------------------------------------------------- databases
class Feature:
    """ov_core::Feature (feat/Feature.h): per-id track container, one camera."""

    def __init__(self, featid: int):
        self.featid = featid
        self.uvs: List[Tuple[float, float]] = []
        self.uvs_norm: List[Tuple[float, float]] = []
        self.timestamps: List[float] = []
        self.chi_test = True     # PL-VIWO's extra flag on ov_core::Feature (Chi_test)


class FeatureDatabase:
    """ov_core::FeatureDatabase::update_feature (feat/FeatureDatabase.cpp:60-85): the sink of the point tracker."""

    def __init__(self):
        self.features_idlookup: Dict[int, Feature] = {}

    def update_feature(self, fid: int, timestamp: float, cam_id: int, u: float, v: float, u_n: float, v_n: float):
        feat = self.features_idlookup.get(fid)
        if feat is None:
            feat = self.features_idlookup[fid] = Feature(fid)
        feat.uvs.append((u, v))
        feat.uvs_norm.append((u_n, v_n))
        feat.timestamps.append(timestamp)

    def get_internal_data(self):
        return self.features_idlookup

    def append_new_measurements(self, database: "FeatureDatabase"):
        """FeatureDatabase::append_new_measurements (feat/FeatureDatabase.cpp:338-387): what UpdaterCamera does with the
        tracker's database right after both trackers ran (UpdaterCamera.cpp:111) — copy the measurements this database
        has not seen yet (matched by timestamp), create unknown features, propagate a failed chi-square flag."""
        for fid, feat in database.get_internal_data().items():
            mine = self.features_idlookup.get(fid)
            if mine is not None:
                if not feat.chi_test:
                    mine.chi_test = False
                    continue
                if not mine.timestamps:
                    mine.timestamps, mine.uvs, mine.uvs_norm = list(feat.timestamps), list(feat.uvs), list(feat.uvs_norm)
                else:
                    seen = list(mine.timestamps)      # the reference searches a COPY taken before appending
                    for i, t in enumerate(feat.timestamps):
                        if t not in seen:
                            mine.timestamps.append(t)
                            mine.uvs.append(feat.uvs[i])
                            mine.uvs_norm.append(feat.uvs_norm[i])
            else:
                new = Feature(feat.featid)
                new.timestamps, new.uvs, new.uvs_norm = list(feat.timestamps), list(feat.uvs), list(feat.uvs_norm)
                new.chi_test = bool(feat.chi_test)
                self.features_idlookup[fid] = new


class LineFeature:
    def __init__(self, featid: int, D: int):
        self.featid = featid
        self.D = D
        self.line_uvs: List[np.ndarray] = []
        self.line_uvs_norm: List[np.ndarray] = []
        self.timestamps: List[float] = []
        self.points: List[int] = []
        self.point_uvs: Dict[float, np.ndarray] = {}


class LineFeatureDatabase:
    """viw::LineFeatureDatabase::update_feature (linefeat/LineFeatureDatabase.cpp:40-76): D is set on creation only."""

    def __init__(self):
        self.features_idlookup: Dict[int, LineFeature] = {}

    def update_feature(self, fid, timestamp, cam_id, line, line_n, points_line: Dict[int, float], points, D):
        feat = self.features_idlookup.get(fid)
        if feat is None:
            feat = self.features_idlookup[fid] = LineFeature(fid, D)
        feat.line_uvs.append(np.asarray(line, np.float32))
        feat.line_uvs_norm.append(np.asarray(line_n, np.float32))
        feat.timestamps.append(timestamp)
        feat.points.extend(points_line.keys())
        feat.point_uvs[timestamp] = np.asarray(points, np.float32)


# ------------------------------------------------------------------------------------------- front end
class FrontEnd:
    """One camera stream: TrackKLT + TrackLSD behind one FeHandle."""

    def __init__(self, cfg: Optional[FeConfig] = None, device: int = 0, camera_model: int = CAM_RADTAN, **kw):
        """camera_model: CAM_RADTAN or CAM_EQUI (cfg.D = k1 k2 k3 k4), fixed for the handle's lifetime."""
        self.cfg = cfg if cfg is not None else default_config(**kw)
        self.camera_model = camera_model
        self._h = C.c_void_p()
        self._lib = lib()
        _check(self._lib.plviwo_fe_create_model(C.byref(self.cfg), camera_model, device, C.byref(self._h)))
        self.database = FeatureDatabase()
        self.line_database = LineFeatureDatabase()
        self.cam_id = 0
        self.info = FeFrameInfo()

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.plviwo_fe_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- reference-shaped calls
    def set_calib(self, K: Sequence[float], D: Sequence[float]):
        _check(self._lib.plviwo_fe_set_calib(self._h, (C.c_double * 4)(*K), (C.c_double * 4)(*D)), self._h)

    def set_num_features(self, n: int):
        _check(self._lib.plviwo_fe_set_num_features(self._h, n), self._h)

    def set_camera(self, model: int, K: Sequence[float], D: Sequence[float]):
        """CamBase model + calibration: the model the handle was created with updates K / D, any other is refused."""
        _check(self._lib.plviwo_fe_set_camera(self._h, model, (C.c_double * 4)(*K), (C.c_double * 4)(*D)), self._h)

    def get_currid(self) -> int:
        v = C.c_uint64(0)
        _check(self._lib.plviwo_fe_get_currid(self._h, C.byref(v)), self._h)
        return int(v.value)

    def set_currid(self, currid: int):
        _check(self._lib.plviwo_fe_set_currid(self._h, currid), self._h)

    def classify_lines(self, vanishing_points):
        """TrackLSD::LineClassification of the last frame's line rows with these vanishing points (3 x (x, y))."""
        vp = (C.c_double * 6)(*np.asarray(vanishing_points, np.float64).reshape(6))
        _check(self._lib.plviwo_fe_classify_lines(self._h, vp), self._h)

    def change_feat_id(self, id_old: int, id_new: int):
        _check(self._lib.plviwo_fe_change_feat_id(self._h, id_old, id_new), self._h)

    def feed_new_camera(self, timestamp: float, image: np.ndarray, mask: Optional[np.ndarray] = None,
                        vanishing_points=None, update_db: bool = True) -> FeFrameInfo:
        """TrackKLT::feed_new_camera followed (when vanishing points are given) by TrackLSD::feed_new_camera, as
        UpdaterCamera::feed_measurement does (UpdaterCamera.cpp:105-110)."""
        if image.dtype != np.uint8 or image.ndim != 2:
            raise FrontEndError(FE_BAD_ARG, "image must be a 2-D uint8 array")
        image = image if image.strides[1] == 1 else np.ascontiguousarray(image)
        mptr, mstride = None, 0
        if mask is not None:
            mask = np.ascontiguousarray(mask, np.uint8)
            mptr, mstride = mask.ctypes.data, mask.strides[0]
        vp = None
        if vanishing_points is not None:
            vp = (C.c_double * 6)(*[float(v) for p in vanishing_points for v in p])
        _check(self._lib.plviwo_fe_feed(self._h, float(timestamp), image.ctypes.data, image.shape[1], image.shape[0],
                                        image.strides[0], mptr, mstride, vp, C.byref(self.info)), self._h)
        if update_db:
            self._push_rows(timestamp)
        return self.info

    def feed_device(self, timestamp: float, d_ptr: int, width: int, height: int, pitch: int, vanishing_points=None):
        vp = None
        if vanishing_points is not None:
            vp = (C.c_double * 6)(*[float(v) for p in vanishing_points for v in p])
        _check(self._lib.plviwo_fe_feed_device(self._h, float(timestamp), d_ptr, width, height, pitch, None, 0, vp,
                                               C.byref(self.info)), self._h)
        return self.info

    def submit(self, timestamp: float, image, stride: int = 0, on_device: bool = False, vanishing_points=None,
               mask: Optional[np.ndarray] = None):
        vp = None
        if vanishing_points is not None:
            vp = (C.c_double * 6)(*[float(v) for p in vanishing_points for v in p])
        if on_device:
            ptr = int(image)
        else:
            ptr, stride = image.ctypes.data, image.strides[0]
        mptr, mstride = None, 0
        if mask is not None:     # the library copies the mask during the call
            mask = np.ascontiguousarray(mask, np.uint8)
            mptr, mstride = mask.ctypes.data, mask.strides[0]
        _check(self._lib.plviwo_fe_submit(self._h, float(timestamp), ptr, stride, 1 if on_device else 0, mptr, mstride, vp), self._h)

    def play(self, timestamps, images, stride: int = 0, on_device: bool = False, vanishing_points=None) -> FePlayStats:
        """Whole-sequence playback inside the library (plviwo_fe_play).  images: list of device pointers (on_device) or of
        2-D uint8 arrays; vanishing_points: per frame 3 x (x, y) or None."""
        n = len(images)
        if on_device:
            ptrs = (C.c_void_p * n)(*[int(p) for p in images])
        else:
            ptrs = (C.c_void_p * n)(*[im.ctypes.data for im in images])
            stride = stride or images[0].strides[0]
        ts = (C.c_double * n)(*[float(t) for t in timestamps])
        vp = None
        if vanishing_points is not None:
            vp = (C.c_double * (6 * n))(*[float(v) for f in vanishing_points for p in f for v in p])
        st = FePlayStats()
        _check(self._lib.plviwo_fe_play(self._h, n, ptrs, stride, 1 if on_device else 0, ts, vp, C.byref(st)), self._h)
        return st

    def collect(self) -> FeFrameInfo:
        _check(self._lib.plviwo_fe_collect(self._h, C.byref(self.info)), self._h)
        return self.info

    def _push_rows(self, timestamp):
        for r in self.point_rows():
            self.database.update_feature(int(r["id"]), timestamp, self.cam_id, float(r["u"]), float(r["v"]),
                                         float(r["un"]), float(r["vn"]))
        lrows, lpts = self.line_rows()
        for r in lrows:
            pts = lpts[r["pt_offset"]:r["pt_offset"] + r["n_pts"]]
            self.line_database.update_feature(int(r["id"]), timestamp, self.cam_id, r["line"], r["line_n"],
                                              {int(p["pid"]): float(p["dist"]) for p in pts},
                                              np.stack([pts["u"], pts["v"]], 1) if len(pts) else np.zeros((0, 2)), int(r["D"]))

    # -- results
    def point_rows(self) -> np.ndarray:
        n = C.c_int(0)
        _check(self._lib.plviwo_fe_get_point_rows(self._h, None, 0, C.byref(n)), self._h)
        out = np.zeros((n.value,), POINT_ROW_DTYPE)
        if n.value:
            _check(self._lib.plviwo_fe_get_point_rows(self._h, out.ctypes.data, n.value, C.byref(n)), self._h)
        return out

    def line_rows(self):
        n = C.c_int(0)
        _check(self._lib.plviwo_fe_get_line_rows(self._h, None, 0, C.byref(n)), self._h)
        rows = np.zeros((n.value,), LINE_ROW_DTYPE)
        if n.value:
            _check(self._lib.plviwo_fe_get_line_rows(self._h, rows.ctypes.data, n.value, C.byref(n)), self._h)
        m = C.c_int(0)
        _check(self._lib.plviwo_fe_get_line_points(self._h, None, 0, C.byref(m)), self._h)
        pts = np.zeros((m.value,), LINE_POINT_DTYPE)
        if m.value:
            _check(self._lib.plviwo_fe_get_line_points(self._h, pts.ctypes.data, m.value, C.byref(m)), self._h)
        return rows, pts

    def line_samples(self):
        n = C.c_int(0)
        _check(self._lib.plviwo_fe_get_line_samples(self._h, None, None, 0, C.byref(n)), self._h)
        uv = np.zeros((n.value, 4), np.float32)
        st = np.zeros((n.value,), np.uint8)
        if n.value:
            _check(self._lib.plviwo_fe_get_line_samples(self._h, uv.ctypes.data, st.ctypes.data, n.value, C.byref(n)), self._h)
        return uv, st

    def get_last_obs(self) -> np.ndarray:
        return self._last()[1]

    def get_last_ids(self) -> np.ndarray:
        return self._last()[0]

    def _last(self):
        n = C.c_int(0)
        _check(self._lib.plviwo_fe_get_last_obs(self._h, None, None, 0, C.byref(n)), self._h)
        ids = np.zeros((n.value,), np.uint64)
        uv = np.zeros((n.value, 2), np.float32)
        if n.value:
            _check(self._lib.plviwo_fe_get_last_obs(self._h, ids.ctypes.data, uv.ctypes.data, n.value, C.byref(n)), self._h)
        return ids, uv

    def get_feature_database(self) -> FeatureDatabase:
        return self.database

    def get_line_feature_database(self) -> LineFeatureDatabase:
        return self.line_database

    # -- state, taps, timing
    def get_state(self) -> bytes:
        n = C.c_size_t(0)
        _check(self._lib.plviwo_fe_get_state(self._h, None, 0, C.byref(n)), self._h)
        buf = C.create_string_buffer(n.value)
        _check(self._lib.plviwo_fe_get_state(self._h, buf, n.value, C.byref(n)), self._h)
        return buf.raw[:n.value]

    def set_state(self, blob: bytes):
        _check(self._lib.plviwo_fe_set_state(self._h, blob, len(blob)), self._h)

    def tap(self, what: int, dtype=np.uint8) -> np.ndarray:
        n = C.c_size_t(0)
        _check(self._lib.plviwo_fe_tap(self._h, what, None, 0, C.byref(n)), self._h)
        out = np.zeros((n.value // np.dtype(dtype).itemsize,), dtype)
        if n.value:
            _check(self._lib.plviwo_fe_tap(self._h, what, out.ctypes.data, n.value, C.byref(n)), self._h)
        return out

    def enable_taps(self, on: bool = True):
        _check(self._lib.plviwo_fe_enable_taps(self._h, 1 if on else 0), self._h)

    def enable_timing(self, on: bool = True):
        _check(self._lib.plviwo_fe_enable_timing(self._h, 1 if on else 0), self._h)

    def stage_times(self, reset: bool = False) -> Dict[str, object]:
        t = FeStageTimes()
        _check(self._lib.plviwo_fe_get_stage_times(self._h, C.byref(t), 1 if reset else 0), self._h)
        return {"ms": {s: t.ms[i] for i, s in enumerate(STAGES)}, "launches": {s: int(t.launches[i]) for i, s in enumerate(STAGES)},
                "frames": int(t.frames), "kernel_launches_total": int(t.kernel_launches_total),
                "h2d_bytes": int(t.h2d_bytes), "d2h_bytes": int(t.d2h_bytes),
                "host_ms": {k: t.host_ms[i] for i, k in enumerate(HOST_STAGES)}}


# ------------------------------------------------------------------------------------------- stream group
class GroupFrontEnd:
    """Many camera streams of one device behind one FeGroupHandle (BASELINE.json configs[4]): stream s is one TrackKLT + one
    TrackLSD; a tick feeds one frame of every stream."""

    def __init__(self, cfg: FeConfig, n_streams: int, device: int = 0, calibs=None, camera_model: int = CAM_RADTAN):
        """camera_model: CAM_RADTAN or CAM_EQUI, one model for every stream, fixed for the group's lifetime."""
        self.cfg = cfg
        self.n = int(n_streams)
        self.camera_model = camera_model
        self._h = C.c_void_p()
        self._lib = lib()
        rc = self._lib.plviwo_fe_group_create_model(C.byref(cfg), self.n, camera_model, device, C.byref(self._h))
        if rc != FE_OK:
            raise FrontEndError(rc, (self._lib.plviwo_fe_group_last_error(None) or b"").decode())
        self.infos = (FeFrameInfo * self.n)()
        if calibs is not None:
            for s, (K, D) in enumerate(calibs):
                self.set_calib(s, K, D)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.plviwo_fe_group_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != FE_OK:
            raise FrontEndError(rc, (self._lib.plviwo_fe_group_last_error(self._h) or b"").decode())

    def set_calib(self, stream: int, K, D):
        self._check(self._lib.plviwo_fe_group_set_calib(self._h, stream, (C.c_double * 4)(*K), (C.c_double * 4)(*D)))

    def set_camera(self, stream: int, model: int, K, D):
        """Calibration with the camera model stated: the group's model updates K / D, any other is refused."""
        self._check(self._lib.plviwo_fe_group_set_camera(self._h, stream, model, (C.c_double * 4)(*K), (C.c_double * 4)(*D)))

    def submit(self, timestamps, images, stride: int = 0, on_device: bool = False, vanishing_points=None, masks=None):
        """images: per stream a 2-D uint8 array / device pointer (on_device) / None (no frame for that stream in this tick);
        vanishing_points: per stream 3 x (x, y), or None (line tracker not fed)."""
        n = self.n
        ptrs = (C.c_void_p * n)()
        keep = []
        for s, im in enumerate(images):
            if im is None:
                ptrs[s] = None
            elif on_device:
                ptrs[s] = int(im)
            else:
                a = im if (im.dtype == np.uint8 and im.strides[1] == 1) else np.ascontiguousarray(im, np.uint8)
                keep.append(a)
                ptrs[s] = a.ctypes.data
                stride = a.strides[0]
        ts = (C.c_double * n)(*[float(t) for t in (timestamps if hasattr(timestamps, "__len__") else [timestamps] * n)])
        vp = None
        if vanishing_points is not None:
            vp = (C.c_double * (6 * n))(*[float(v) for f in vanishing_points for p in f for v in p])
        mp, mstride = None, 0
        if masks is not None:
            mp = (C.c_void_p * n)()
            for s, m in enumerate(masks):
                if m is None:
                    mp[s] = None
                else:
                    a = np.ascontiguousarray(m, np.uint8)
                    keep.append(a)
                    mp[s] = a.ctypes.data
                    mstride = a.strides[0]
        self._check(self._lib.plviwo_fe_group_submit(self._h, ts, ptrs, stride, 1 if on_device else 0, mp, mstride, vp))

    def collect(self):
        self._check(self._lib.plviwo_fe_group_collect(self._h, self.infos))
        return self.infos

    def feed(self, timestamps, images, vanishing_points=None, masks=None):
        self.submit(timestamps, images, vanishing_points=vanishing_points, masks=masks)
        return self.collect()

    def play(self, timestamps, ptr_table, stride: int, on_device: bool, vanishing_points=None):
        """ptr_table: ctypes array of n_ticks * n_streams pointers (tick-major); vanishing_points: per stream 3 x (x, y)."""
        n_ticks = len(timestamps)
        ts = (C.c_double * n_ticks)(*[float(t) for t in timestamps])
        vp = None
        if vanishing_points is not None:
            vp = (C.c_double * (6 * self.n))(*[float(v) for f in vanishing_points for p in f for v in p])
        st = (FePlayStats * self.n)()
        self._check(self._lib.plviwo_fe_group_play(self._h, n_ticks, ptr_table, stride, 1 if on_device else 0, ts, vp, st))
        return st

    def _rows(self, fn, stream, dtype):
        n = C.c_int(0)
        self._check(fn(self._h, stream, None, 0, C.byref(n)))
        out = np.zeros((n.value,), dtype)
        if n.value:
            self._check(fn(self._h, stream, out.ctypes.data, n.value, C.byref(n)))
        return out

    def point_rows(self, stream: int) -> np.ndarray:
        return self._rows(self._lib.plviwo_fe_group_get_point_rows, stream, POINT_ROW_DTYPE)

    def line_rows(self, stream: int):
        return (self._rows(self._lib.plviwo_fe_group_get_line_rows, stream, LINE_ROW_DTYPE),
                self._rows(self._lib.plviwo_fe_group_get_line_points, stream, LINE_POINT_DTYPE))

    def last_obs(self, stream: int):
        n = C.c_int(0)
        self._check(self._lib.plviwo_fe_group_get_last_obs(self._h, stream, None, None, 0, C.byref(n)))
        ids = np.zeros((n.value,), np.uint64)
        uv = np.zeros((n.value, 2), np.float32)
        if n.value:
            self._check(self._lib.plviwo_fe_group_get_last_obs(self._h, stream, ids.ctypes.data, uv.ctypes.data, n.value, C.byref(n)))
        return ids, uv

    def line_samples(self, stream: int):
        """cfg.line_samples: the samples of stream `stream` in the last collected tick, as FrontEnd.line_samples():
        uv (n, 4) float32 = u0 v0 (previous image) u1 v1 (current image), status (n,) uint8."""
        n = C.c_int(0)
        self._check(self._lib.plviwo_fe_group_get_line_samples(self._h, stream, None, None, 0, C.byref(n)))
        uv = np.zeros((n.value, 4), np.float32)
        st = np.zeros((n.value,), np.uint8)
        if n.value:
            self._check(self._lib.plviwo_fe_group_get_line_samples(self._h, stream, uv.ctypes.data, st.ctypes.data, n.value,
                                                                   C.byref(n)))
        return uv, st

    def get_state(self, stream: int) -> bytes:
        n = C.c_size_t(0)
        self._check(self._lib.plviwo_fe_group_get_state(self._h, stream, None, 0, C.byref(n)))
        buf = C.create_string_buffer(n.value)
        self._check(self._lib.plviwo_fe_group_get_state(self._h, stream, buf, n.value, C.byref(n)))
        return buf.raw[:n.value]

    def set_state(self, stream: int, blob: bytes):
        self._check(self._lib.plviwo_fe_group_set_state(self._h, stream, blob, len(blob)))

    def tap(self, stream: int, what: int) -> np.ndarray:
        n = C.c_size_t(0)
        self._check(self._lib.plviwo_fe_group_tap(self._h, stream, what, None, 0, C.byref(n)))
        out = np.zeros((n.value,), np.uint8)
        if n.value:
            self._check(self._lib.plviwo_fe_group_tap(self._h, stream, what, out.ctypes.data, n.value, C.byref(n)))
        return out

    def enable_timing(self, on: bool = True):
        self._check(self._lib.plviwo_fe_group_enable_timing(self._h, 1 if on else 0))

    def times(self, reset: bool = False) -> Dict[str, object]:
        t = FeGroupTimes()
        self._check(self._lib.plviwo_fe_group_get_times(self._h, C.byref(t), 1 if reset else 0))
        return {"ms": {k: t.ms[i] for i, k in enumerate(GROUP_KERNELS)}, "launches": {k: int(t.launches[i]) for i, k in enumerate(GROUP_KERNELS)},
                "frames_of": {k: int(t.frames[i]) for i, k in enumerate(GROUP_KERNELS)}, "ticks": int(t.ticks),
                "frames": int(t.frames_total), "kernel_launches_total": int(t.kernel_launches_total),
                "h2d_bytes": int(t.h2d_bytes), "d2h_bytes": int(t.d2h_bytes), "fast_cells": int(t.fast_cells)}


class StereoGroupFrontEnd:
    """Many stereo rigs of one device behind one FeStereoGroupHandle: rig r is what one StereoFrontEnd is (same rows, bit for
    bit); a tick feeds one stereo pair of every rig.  Cameras: 0 left, 1 right."""

    def __init__(self, cfg: FeConfig, n_rigs: int, device: int = 0, calibs=None, camera_model: int = CAM_RADTAN):
        """calibs: per rig ((K_left, D_left), (K_right, D_right)), or None (cfg.K / cfg.D for every camera).  camera_model:
        CAM_RADTAN or CAM_EQUI, one model for every camera, fixed for the group's lifetime."""
        self.cfg = cfg
        self.n = int(n_rigs)
        self.camera_model = camera_model
        self._h = C.c_void_p()
        self._lib = lib()
        rc = self._lib.plviwo_fe_stereo_group_create_model(C.byref(cfg), self.n, camera_model, device, C.byref(self._h))
        if rc != FE_OK:
            raise FrontEndError(rc, (self._lib.plviwo_fe_stereo_group_last_error(None) or b"").decode())
        self.infos = (FeStereoInfo * self.n)()
        if calibs is not None:
            for r, cams in enumerate(calibs):
                for cam, (K, D) in enumerate(cams):
                    self.set_calib(r, cam, K, D)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.plviwo_fe_stereo_group_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != FE_OK:
            raise FrontEndError(rc, (self._lib.plviwo_fe_stereo_group_last_error(self._h) or b"").decode())

    def set_calib(self, rig: int, cam: int, K, D):
        self._check(self._lib.plviwo_fe_stereo_group_set_calib(self._h, rig, cam, (C.c_double * 4)(*K), (C.c_double * 4)(*D)))

    def set_camera(self, rig: int, cam: int, model: int, K, D):
        """Calibration with the camera model stated: the group's model updates K / D, any other is refused."""
        self._check(self._lib.plviwo_fe_stereo_group_set_camera(self._h, rig, cam, model, (C.c_double * 4)(*K), (C.c_double * 4)(*D)))

    def _ptrs(self, arrays, keep, on_device=False):
        out = (C.c_void_p * self.n)()
        stride = 0
        for r, im in enumerate(arrays):
            if im is None:
                out[r] = None
            elif on_device:
                out[r] = int(im)
            else:
                a = im if (im.dtype == np.uint8 and im.strides[1] == 1) else np.ascontiguousarray(im, np.uint8)
                keep.append(a)
                out[r] = a.ctypes.data
                stride = a.strides[0]
        return out, stride

    def submit(self, timestamps, pairs, stride: int = 0, on_device: bool = False, vanishing_points=None, masks=None):
        """pairs: per rig (left, right) 2-D uint8 arrays / device pointers (on_device), or None (no pair for that rig in this
        tick); vanishing_points: per rig 3 x (x, y), or None (line tracker not fed); masks: per rig (left, right) or None."""
        keep = []
        pl, s0 = self._ptrs([None if p is None else p[0] for p in pairs], keep, on_device)
        pr, s1 = self._ptrs([None if p is None else p[1] for p in pairs], keep, on_device)
        stride = stride or s0 or s1
        ts = (C.c_double * self.n)(*[float(t) for t in (timestamps if hasattr(timestamps, "__len__") else [timestamps] * self.n)])
        vp = None
        if vanishing_points is not None:
            vp = (C.c_double * (6 * self.n))(*[float(v) for f in vanishing_points for p in f for v in p])
        ml = mr = None
        mstride = 0
        if masks is not None:
            ml, mstride = self._ptrs([None if m is None else m[0] for m in masks], keep)
            mr, _ = self._ptrs([None if m is None else m[1] for m in masks], keep)
        self._check(self._lib.plviwo_fe_stereo_group_submit(self._h, ts, pl, pr, stride, 1 if on_device else 0, ml, mr, mstride, vp))

    def collect(self):
        self._check(self._lib.plviwo_fe_stereo_group_collect(self._h, self.infos))
        return self.infos

    def feed(self, timestamps, pairs, vanishing_points=None, masks=None):
        self.submit(timestamps, pairs, vanishing_points=vanishing_points, masks=masks)
        return self.collect()

    def play(self, timestamps, ptr_table, stride: int, on_device: bool, vanishing_points=None):
        """ptr_table: ctypes array of n_ticks * n_rigs * 2 pointers, [(t * n_rigs + r) * 2 + cam]; vanishing_points: per rig."""
        n_ticks = len(timestamps)
        ts = (C.c_double * n_ticks)(*[float(t) for t in timestamps])
        vp = None
        if vanishing_points is not None:
            vp = (C.c_double * (6 * self.n))(*[float(v) for f in vanishing_points for p in f for v in p])
        st = (FePlayStats * self.n)()
        self._check(self._lib.plviwo_fe_stereo_group_play(self._h, n_ticks, ptr_table, stride, 1 if on_device else 0, ts, vp, st))
        return st

    def _rows(self, fn, args, dtype):
        n = C.c_int(0)
        self._check(fn(self._h, *args, None, 0, C.byref(n)))
        out = np.zeros((n.value,), dtype)
        if n.value:
            self._check(fn(self._h, *args, out.ctypes.data, n.value, C.byref(n)))
        return out

    def point_rows(self, rig: int, cam: int) -> np.ndarray:
        return self._rows(self._lib.plviwo_fe_stereo_group_get_point_rows, (rig, cam), POINT_ROW_DTYPE)

    def line_rows(self, rig: int):
        """Line rows and line points of the rig's left image."""
        return (self._rows(self._lib.plviwo_fe_stereo_group_get_line_rows, (rig,), LINE_ROW_DTYPE),
                self._rows(self._lib.plviwo_fe_stereo_group_get_line_points, (rig,), LINE_POINT_DTYPE))

    def last_obs(self, rig: int, cam: int):
        n = C.c_int(0)
        self._check(self._lib.plviwo_fe_stereo_group_get_last_obs(self._h, rig, cam, None, None, 0, C.byref(n)))
        ids = np.zeros((n.value,), np.uint64)
        uv = np.zeros((n.value, 2), np.float32)
        if n.value:
            self._check(self._lib.plviwo_fe_stereo_group_get_last_obs(self._h, rig, cam, ids.ctypes.data, uv.ctypes.data, n.value,
                                                                      C.byref(n)))
        return ids, uv

    def get_state(self, rig: int) -> bytes:
        n = C.c_size_t(0)
        self._check(self._lib.plviwo_fe_stereo_group_get_state(self._h, rig, None, 0, C.byref(n)))
        buf = C.create_string_buffer(n.value)
        self._check(self._lib.plviwo_fe_stereo_group_get_state(self._h, rig, buf, n.value, C.byref(n)))
        return buf.raw[:n.value]

    def set_state(self, rig: int, blob: bytes):
        self._check(self._lib.plviwo_fe_stereo_group_set_state(self._h, rig, blob, len(blob)))


class GroupEngine:
    """bench.py adapter: the streams of one rank behind one stream group, driven through plviwo_fe_group_play (the
    submit / collect loop inside the library)."""
    name = "group"

    def __init__(self, fe_mod, dev, metas, workload, lookahead=None):
        # ticks in flight: the chain walk of a tick's frames lasts ~3 ms (its longest component), the other kernels of a tick
        # ~2 ms: six ticks in flight keep the device busy while walks finish (measured: 3 -> 6 ticks +5 %, 10 no more)
        # (profiles/sweep_group.sh, one B200: 64 streams 3 ticks 31.7 k frames/s, 6: 33.6 k, 12: 38.3 k, 16: 38.6 k; 8 streams
        # 12: 15.1 k, 24: 20.2 k, 48: 20.1 k)
        # after FAST moved on demand and the line association came off the point chain (round 2, second half): 64 streams, 12 / 24 /
        # 36 ticks in flight: 47.8 k / 49.3 k / 49.7 k frames/s
        la = int(os.environ.get("PLVIWO_BENCH_GROUP_LA", "0")) or lookahead or 24
        self.lookahead = la
        self.metas = metas
        self.g = GroupFrontEnd(default_config(lookahead=la, **workload), len(metas), device=dev, calibs=[(K, D) for K, D, _ in metas])

    def run(self, first, n_frames, ptrs, pitch, on_device, frame_index=None):
        S = len(self.metas)
        fi = frame_index or (lambda i: i)
        tab = (C.c_void_p * (n_frames * S))()
        for i in range(n_frames):
            t = fi(first + i)
            for k in range(S):
                p = ptrs[k][t]
                tab[i * S + k] = int(p) if on_device else p.ctypes.data
        ts = [1.0 + 0.1 * (first + i) for i in range(n_frames)]
        # PLVIWO_BENCH_NO_LINES=1 (experiments only): the line tracker is not fed, the point path runs alone
        vps = None if os.environ.get("PLVIWO_BENCH_NO_LINES") else [m[2] for m in self.metas]
        st = self.g.play(ts, tab, pitch, on_device, vanishing_points=vps)
        return int(sum(x.frames for x in st))

    def counters(self, reset=False):
        t = self.g.times(reset=reset)
        return {k: t[k] for k in ("kernel_launches_total", "h2d_bytes", "d2h_bytes", "frames")}

    def stage_times(self, reset=False):
        return {"group": self.g.times(reset=reset)}

    def enable_timing(self, on):
        self.g.enable_timing(on)

    def close(self):
        self.g.close()


# ------------------------------------------------------------------------------------------- tracker state blob
_STATE_MAGIC = 0x504C5657
_STATE_HDR = np.dtype([("magic", "<u4"), ("version", "<u4"), ("w", "<i4"), ("h", "<i4"), ("currid", "<u8"),
                       ("line_currid", "<u8"), ("n_pts", "<i4"), ("n_lines", "<i4"), ("has_image", "<i4"),
                       ("has_mask", "<i4"), ("n_pol", "<i4"), ("reserved", "<i4")])


class StereoFrontEnd:
    """One stereo rig: ov_core::TrackKLT with use_stereo = true behind one FeStereoHandle (camera 0 = left, 1 = right)."""

    def __init__(self, cfg: Optional[FeConfig] = None, K_right=None, D_right=None, device: int = 0, camera_model: int = CAM_RADTAN,
                 **kw):
        """camera_model: CAM_RADTAN or CAM_EQUI for both cameras, fixed for the rig's lifetime."""
        self.cfg = cfg if cfg is not None else default_config(**kw)
        self.camera_model = camera_model
        self._h = C.c_void_p()
        self._lib = lib()
        kr = None if K_right is None else (C.c_double * 4)(*K_right)
        dr = None if D_right is None else (C.c_double * 4)(*D_right)
        rc = self._lib.plviwo_fe_stereo_create_model(C.byref(self.cfg), camera_model, kr, dr, device, C.byref(self._h))
        if rc != FE_OK:
            raise FrontEndError(rc, (self._lib.plviwo_fe_stereo_last_error(None) or b"").decode())
        self.database = FeatureDatabase()      # one database shared by both cameras (UpdaterCamera.cpp:47-56)
        self.line_database = LineFeatureDatabase()
        self.info = FeStereoInfo()

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.plviwo_fe_stereo_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != FE_OK:
            raise FrontEndError(rc, (self._lib.plviwo_fe_stereo_last_error(self._h) or b"").decode())

    def set_calib(self, cam: int, K, D):
        self._check(self._lib.plviwo_fe_stereo_set_calib(self._h, cam, (C.c_double * 4)(*K), (C.c_double * 4)(*D)))

    def set_camera(self, cam: int, model: int, K, D):
        """Calibration with the camera model stated: the rig's model updates K / D, any other is refused."""
        self._check(self._lib.plviwo_fe_stereo_set_camera(self._h, cam, model, (C.c_double * 4)(*K), (C.c_double * 4)(*D)))

    def set_num_features(self, n: int):
        self._check(self._lib.plviwo_fe_stereo_set_num_features(self._h, n))

    def change_feat_id(self, id_old: int, id_new: int):
        self._check(self._lib.plviwo_fe_stereo_change_feat_id(self._h, id_old, id_new))

    @staticmethod
    def _img(a):
        if a.dtype != np.uint8 or a.ndim != 2:
            raise FrontEndError(FE_BAD_ARG, "image must be a 2-D uint8 array")
        return np.ascontiguousarray(a)

    @staticmethod
    def _vp(vanishing_points):
        if vanishing_points is None:
            return None
        return (C.c_double * 6)(*[float(v) for p in vanishing_points for v in p])

    def feed_new_camera(self, timestamp: float, image_left, image_right, mask_left=None, mask_right=None,
                        vanishing_points=None, update_db: bool = True) -> FeStereoInfo:
        """TrackKLT::feed_new_camera with a two-image message (TrackKLT.cpp:34-94 -> feed_stereo), followed (when
        vanishing points are given and cfg.use_lines) by TrackLSD::feed_new_camera, which takes the left image
        (TrackLSD.cpp:57-60)."""
        il, ir = self._img(image_left), self._img(image_right)
        if il.shape != ir.shape:
            raise FrontEndError(FE_BAD_ARG, "left and right image sizes differ")
        ml = None if mask_left is None else np.ascontiguousarray(mask_left, np.uint8)
        mr = None if mask_right is None else np.ascontiguousarray(mask_right, np.uint8)
        self._check(self._lib.plviwo_fe_stereo_feed(
            self._h, float(timestamp), il.ctypes.data, ir.ctypes.data, il.shape[1], il.shape[0], il.strides[0],
            None if ml is None else ml.ctypes.data, None if mr is None else mr.ctypes.data, il.shape[1],
            self._vp(vanishing_points), C.byref(self.info)))
        if update_db:
            self._push_rows(timestamp)
        return self.info

    def submit(self, timestamp: float, image_left, image_right, stride: int = 0, on_device: bool = False, vanishing_points=None):
        """image_*: numpy arrays (host) or integer device pointers (on_device, with stride)."""
        if on_device:
            pl, pr = int(image_left), int(image_right)
        else:
            pl, pr, stride = image_left.ctypes.data, image_right.ctypes.data, image_left.strides[0]
        self._check(self._lib.plviwo_fe_stereo_submit(self._h, float(timestamp), pl, pr, stride, 1 if on_device else 0, None, None, 0,
                                                      self._vp(vanishing_points)))

    def collect(self) -> FeStereoInfo:
        self._check(self._lib.plviwo_fe_stereo_collect(self._h, C.byref(self.info)))
        return self.info

    def _push_rows(self, timestamp):
        for cam in (0, 1):    # left rows first, then right (TrackKLT.cpp:352-363)
            for r in self.point_rows(cam):
                self.database.update_feature(int(r["id"]), timestamp, cam, float(r["u"]), float(r["v"]), float(r["un"]), float(r["vn"]))
        lrows, lpts = self.line_rows()
        for r in lrows:
            pts = lpts[r["pt_offset"]:r["pt_offset"] + r["n_pts"]]
            self.line_database.update_feature(int(r["id"]), timestamp, 0, r["line"], r["line_n"],
                                              {int(p["pid"]): float(p["dist"]) for p in pts},
                                              np.stack([pts["u"], pts["v"]], 1) if len(pts) else np.zeros((0, 2)), int(r["D"]))

    def line_rows(self):
        n = C.c_int(0)
        self._check(self._lib.plviwo_fe_stereo_get_line_rows(self._h, None, 0, C.byref(n)))
        rows = np.zeros((n.value,), LINE_ROW_DTYPE)
        if n.value:
            self._check(self._lib.plviwo_fe_stereo_get_line_rows(self._h, rows.ctypes.data, n.value, C.byref(n)))
        m = C.c_int(0)
        self._check(self._lib.plviwo_fe_stereo_get_line_points(self._h, None, 0, C.byref(m)))
        pts = np.zeros((m.value,), LINE_POINT_DTYPE)
        if m.value:
            self._check(self._lib.plviwo_fe_stereo_get_line_points(self._h, pts.ctypes.data, m.value, C.byref(m)))
        return rows, pts

    def classify_lines(self, vanishing_points):
        self._check(self._lib.plviwo_fe_stereo_classify_lines(self._h, self._vp(vanishing_points)))

    def point_rows(self, cam: int) -> np.ndarray:
        n = C.c_int(0)
        self._check(self._lib.plviwo_fe_stereo_get_point_rows(self._h, cam, None, 0, C.byref(n)))
        out = np.zeros((n.value,), POINT_ROW_DTYPE)
        if n.value:
            self._check(self._lib.plviwo_fe_stereo_get_point_rows(self._h, cam, out.ctypes.data, n.value, C.byref(n)))
        return out

    def _last(self, cam: int):
        n = C.c_int(0)
        self._check(self._lib.plviwo_fe_stereo_get_last_obs(self._h, cam, None, None, 0, C.byref(n)))
        ids = np.zeros((n.value,), np.uint64)
        uv = np.zeros((n.value, 2), np.float32)
        if n.value:
            self._check(self._lib.plviwo_fe_stereo_get_last_obs(self._h, cam, ids.ctypes.data, uv.ctypes.data, n.value, C.byref(n)))
        return ids, uv

    def get_last_obs(self):
        return {cam: self._last(cam)[1] for cam in (0, 1)}

    def get_last_ids(self):
        return {cam: self._last(cam)[0] for cam in (0, 1)}

    def get_feature_database(self) -> FeatureDatabase:
        return self.database

    def get_state(self) -> bytes:
        n = C.c_size_t(0)
        self._check(self._lib.plviwo_fe_stereo_get_state(self._h, None, 0, C.byref(n)))
        buf = C.create_string_buffer(n.value)
        self._check(self._lib.plviwo_fe_stereo_get_state(self._h, buf, n.value, C.byref(n)))
        return buf.raw[:n.value]

    def set_state(self, blob: bytes):
        self._check(self._lib.plviwo_fe_stereo_set_state(self._h, blob, len(blob)))

    def stage_times(self, reset: bool = False) -> Dict[str, object]:
        t = FeStageTimes()
        self._check(self._lib.plviwo_fe_stereo_get_stage_times(self._h, C.byref(t), 1 if reset else 0))
        return {"frames": int(t.frames), "kernel_launches_total": int(t.kernel_launches_total), "h2d_bytes": int(t.h2d_bytes),
                "d2h_bytes": int(t.d2h_bytes)}


_STEREO_HDR = np.dtype([("magic", "<u4"), ("version", "<u4"), ("currid", "<u8"), ("size", "<u8", (2,))])


def pack_stereo_state(currid: int, blob_left: bytes, blob_right: bytes) -> bytes:
    """Stereo state blob: header + one monocular blob (pack_state) per camera; the per-camera currid fields are ignored."""
    hdr = np.zeros((), _STEREO_HDR)
    hdr["magic"], hdr["version"], hdr["currid"] = 0x504C5653, 1, currid
    hdr["size"] = (len(blob_left), len(blob_right))
    return hdr.tobytes() + blob_left + blob_right


def unpack_stereo_state(blob: bytes):
    hdr = np.frombuffer(blob, _STEREO_HDR, 1)[0]
    o = _STEREO_HDR.itemsize
    a, b = int(hdr["size"][0]), int(hdr["size"][1])
    return int(hdr["currid"]), unpack_state(blob[o:o + a]), unpack_state(blob[o + a:o + a + b])


def pack_state(width, height, currid, pts_last, ids_last, img_last_eq=None, mask_last=None, line_currid=1,
               lines_last=None, line_ids_last=None, pol_last=None) -> bytes:
    """Serialises tracker state in the layout plviwo_fe_set_state expects (teacher forcing / resume):
    TrackBase members pts_last / ids_last / currid / img_last (equalised) / img_mask_last and TrackLSD members
    lines_last / ids_last / point_on_lines_last / currid."""
    pts = np.ascontiguousarray(pts_last, np.float32).reshape(-1, 2)
    ids = np.ascontiguousarray(ids_last, np.uint64).reshape(-1)
    lines = np.zeros((0, 4), np.float32) if lines_last is None else np.ascontiguousarray(lines_last, np.float32).reshape(-1, 4)
    lids = np.zeros((0,), np.uint64) if line_ids_last is None else np.ascontiguousarray(line_ids_last, np.uint64).reshape(-1)
    pol = [] if pol_last is None else pol_last
    hdr = np.zeros((), _STATE_HDR)
    hdr["magic"], hdr["version"], hdr["w"], hdr["h"] = _STATE_MAGIC, 1, width, height
    hdr["currid"], hdr["line_currid"] = currid, line_currid
    hdr["n_pts"], hdr["n_lines"] = len(pts), len(lines)
    hdr["has_image"] = 0 if img_last_eq is None else 1
    hdr["has_mask"] = 0 if (mask_last is None or img_last_eq is None or not np.any(mask_last)) else 1
    hdr["n_pol"] = sum(len(m) for m in pol)
    parts = [hdr.tobytes(), pts.tobytes(), ids.tobytes(), lines.tobytes(), lids.tobytes(),
             np.array([len(m) for m in pol], np.int32).tobytes()]
    ent = np.zeros((int(hdr["n_pol"]),), np.dtype([("k", "<i4"), ("v", "<f8")], align=False))
    i = 0
    for m in pol:
        for k in sorted(m):
            ent[i] = (k, m[k])
            i += 1
    parts.append(ent.tobytes())
    if img_last_eq is not None:
        parts.append(np.ascontiguousarray(img_last_eq, np.uint8).tobytes())
        if hdr["has_mask"]:
            parts.append(np.ascontiguousarray(mask_last, np.uint8).tobytes())
    return b"".join(parts)


def unpack_state(blob: bytes) -> Dict[str, object]:
    hdr = np.frombuffer(blob, _STATE_HDR, 1)[0]
    o = _STATE_HDR.itemsize
    n, m = int(hdr["n_pts"]), int(hdr["n_lines"])
    pts = np.frombuffer(blob, np.float32, 2 * n, o).reshape(-1, 2); o += 8 * n
    ids = np.frombuffer(blob, np.uint64, n, o); o += 8 * n
    lines = np.frombuffer(blob, np.float32, 4 * m, o).reshape(-1, 4); o += 16 * m
    lids = np.frombuffer(blob, np.uint64, m, o); o += 8 * m
    sizes = np.frombuffer(blob, np.int32, m, o); o += 4 * m
    ent = np.frombuffer(blob, np.dtype([("k", "<i4"), ("v", "<f8")], align=False), int(hdr["n_pol"]), o)
    o += 12 * int(hdr["n_pol"])
    pol, e = [], 0
    for sz in sizes:
        pol.append({int(ent[e + j]["k"]): float(ent[e + j]["v"]) for j in range(sz)})
        e += sz
    w, h = int(hdr["w"]), int(hdr["h"])
    img = mask = None
    if hdr["has_image"]:
        img = np.frombuffer(blob, np.uint8, w * h, o).reshape(h, w); o += w * h
        if hdr["has_mask"]:
            mask = np.frombuffer(blob, np.uint8, w * h, o).reshape(h, w)
    return dict(currid=int(hdr["currid"]), line_currid=int(hdr["line_currid"]), pts_last=pts, ids_last=ids, lines_last=lines,
                line_ids_last=lids, pol_last=pol, img_last=img, mask_last=mask)


# ------------------------------------------------------------------------------------------- stand-alone ops
def pyramid_level_sizes(w: int, h: int, levels: int):
    out = []
    for _ in range(levels + 1):
        out.append((w, h))
        w, h = (w + 1) // 2, (h + 1) // 2
        if w < 2 or h < 2:
            break
    return out


def op_equalize_pyramid(img: np.ndarray, levels: int, device: int = 0):
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    sizes = pyramid_level_sizes(w, h, levels)
    out = np.zeros((sum(a * b for a, b in sizes),), np.uint8)
    half = np.zeros((h // 2, w // 2), np.uint8)
    _check(lib().plviwo_op_equalize_pyramid(device, img.ctypes.data, w, h, levels, out.ctypes.data, half.ctypes.data))
    lv, o = [], 0
    for (lw, lh) in sizes:
        lv.append(out[o:o + lw * lh].reshape(lh, lw))
        o += lw * lh
    return lv, half


def op_clahe(img: np.ndarray, device: int = 0) -> np.ndarray:
    img = np.ascontiguousarray(img, np.uint8)
    out = np.empty_like(img)
    _check(lib().plviwo_op_clahe(device, img.ctypes.data, img.shape[1], img.shape[0], out.ctypes.data))
    return out


def op_fast_cell(img: np.ndarray, threshold: int, device: int = 0) -> np.ndarray:
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    cap = w * h // 4 + 16
    out = np.zeros((cap, 3), np.int32)
    n = C.c_int(0)
    _check(lib().plviwo_op_fast_cell(device, img.ctypes.data, w, h, threshold, out.ctypes.data, cap, C.byref(n)))
    return out[:n.value].copy()


def op_sort_corners(packed: np.ndarray, nfg: int, device: int = -1, prefix: bool = False):
    """Grider_GRID.h:128-133 on packed corners (x | y << 12 | score << 24).  device < 0: host instantiation, returns the
    whole sorted list; device >= 0: the selection kernel, returns the (x, y) of the first nfg."""
    packed = np.ascontiguousarray(packed, np.uint32)
    n = C.c_int(0)
    if device < 0:
        out = np.empty_like(packed)
        pre = np.zeros((nfg, 2), np.float32)
        _check(lib().plviwo_op_sort_corners(device, packed.ctypes.data, len(packed), nfg, out.ctypes.data, pre.ctypes.data, C.byref(n)))
        if prefix:
            return out, pre[:n.value]
        return out
    cand = np.zeros((nfg, 2), np.float32)
    _check(lib().plviwo_op_sort_corners(device, packed.ctypes.data, len(packed), nfg, None, cand.ctypes.data, C.byref(n)))
    return cand[:n.value]


def op_corner_subpix(img: np.ndarray, pts: np.ndarray, device: int = 0) -> np.ndarray:
    img = np.ascontiguousarray(img, np.uint8)
    p = np.ascontiguousarray(pts, np.float32).reshape(-1, 2).copy()
    _check(lib().plviwo_op_corner_subpix(device, img.ctypes.data, img.shape[1], img.shape[0], p.ctypes.data, len(p)))
    return p


def op_lk(img0, img1, pts0, pts1_init, win: int = 15, max_level: int = 5, device: int = 0, form: str = "cta"):
    """calcOpticalFlowPyrLK with an initial flow.  form "cta": the single-handle kernels (k_lk15 for win 15); "warp": the
    stream group's one-warp-per-feature kernel (win 15, max_level <= 5), which gives the same results bit for bit."""
    if form not in ("cta", "warp"):
        raise ValueError("form must be 'cta' or 'warp', not %r" % (form,))
    img0 = np.ascontiguousarray(img0, np.uint8)
    img1 = np.ascontiguousarray(img1, np.uint8)
    p0 = np.ascontiguousarray(pts0, np.float32).reshape(-1, 2)
    p1 = np.ascontiguousarray(pts1_init, np.float32).reshape(-1, 2).copy()
    st = np.zeros((len(p0),), np.uint8)
    fn = lib().plviwo_op_lk if form == "cta" else lib().plviwo_op_lk_warp
    _check(fn(device, img0.ctypes.data, img1.ctypes.data, img0.shape[1], img0.shape[0], win, max_level,
              p0.ctypes.data, p1.ctypes.data, st.ctypes.data, len(p0)))
    return p1, st


def op_undistort(pts, K, D, device: int = 0) -> np.ndarray:
    p = np.ascontiguousarray(pts, np.float32).reshape(-1, 2)
    out = np.zeros_like(p)
    _check(lib().plviwo_op_undistort(device, p.ctypes.data, len(p), (C.c_double * 4)(*K), (C.c_double * 4)(*D), out.ctypes.data))
    return out


def op_undistort_equi(pts, K, D, device: int = 0) -> np.ndarray:
    """cv::fisheye::undistortPoints of (n, 2) points; device < 0 runs the host instantiation of the same arithmetic."""
    p = np.ascontiguousarray(pts, np.float32).reshape(-1, 2)
    out = np.zeros_like(p)
    _check(lib().plviwo_op_undistort_equi(device, p.ctypes.data, len(p), (C.c_double * 4)(*K), (C.c_double * 4)(*D), out.ctypes.data))
    return out


def op_canny(img: np.ndarray, th: float = 50.0, device: int = 0) -> np.ndarray:
    img = np.ascontiguousarray(img, np.uint8)
    out = np.zeros_like(img)
    _check(lib().plviwo_op_canny_half(device, img.ctypes.data, img.shape[1], img.shape[0], th, out.ctypes.data))
    return out


def op_ccl_tiles(edges: np.ndarray, device: int = 0) -> Dict[str, np.ndarray]:
    """Connected components of every 64 x 16 tile of an edge map (h x w, nonzero = edge) on their own: label (h x w,
    raster index of the tile-local root, -1 off the edges), cnt and bbox (3 x h x w; meaningful at the roots) and the
    sorted tile-local roots."""
    e = np.ascontiguousarray(edges) != 0
    h, w = e.shape
    wpr = (w + 31) // 32
    padded = np.zeros((h, wpr * 32), bool)
    padded[:, :w] = e
    words = np.ascontiguousarray(np.packbits(padded, axis=1, bitorder="little").view("<u4"))
    label = np.empty((h, w), np.int32)
    cnt = np.empty((h, w), np.int32)
    bbox = np.empty((3, h, w), np.int32)
    cap = w * h // 4 + 1
    roots = np.empty(cap, np.int32)
    n = C.c_int(0)
    _check(lib().plviwo_op_ccl_tiles(device, words.ctypes.data, w, h, label.ctypes.data, cnt.ctypes.data, bbox.ctypes.data,
                                     roots.ctypes.data, cap, C.byref(n)))
    return {"label": label, "cnt": cnt, "bbox": bbox, "roots": np.sort(roots[:n.value])}


def op_fld(img: np.ndarray, length_threshold: int = 20, distance_threshold: float = 1.414213562, canny_th: float = 50.0,
           device: int = 0) -> np.ndarray:
    img = np.ascontiguousarray(img, np.uint8)
    cap = 8192
    out = np.zeros((cap, 4), np.float32)
    n = C.c_int(0)
    _check(lib().plviwo_op_fld(device, img.ctypes.data, img.shape[1], img.shape[0], length_threshold, distance_threshold,
                               canny_th, out.ctypes.data, cap, C.byref(n)))
    return out[:n.value].copy()


def op_image_kernels_time(w: int, h: int, iters: int = 10, device: int = 0) -> Dict[str, float]:
    """Mean ms per launch of k_hist, k_eq_pyr1, k_fast, k_canny on a device-resident w x h image (micro-benchmark)."""
    ms = (C.c_float * 4)()
    _check(lib().plviwo_op_image_kernels_time(device, w, h, iters, ms))
    return {"hist": ms[0], "eq_pyr1": ms[1], "fast": ms[2], "canny": ms[3]}


def op_assign_points(lines, points, pids):
    """TrackLSD::AssignPointToLines through the library's host implementation: returns (kept line indices,
    [{point id: distance}] per kept line)."""
    ln = np.ascontiguousarray(lines, np.float32).reshape(-1, 4)
    pt = np.ascontiguousarray(points, np.float32).reshape(-1, 2)
    pid = np.ascontiguousarray(pids, np.uint64).reshape(-1)
    kept = np.zeros(len(ln), np.int32)
    off = np.zeros(len(ln) + 1, np.int32)
    cap = max(len(ln) * max(len(pt), 1), 1)
    po = np.zeros(cap, np.int32)
    do = np.zeros(cap, np.float32)
    n = C.c_int(0)
    L = lib()
    L.plviwo_op_assign_points.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_int, C.POINTER(C.c_int)]
    _check(L.plviwo_op_assign_points(len(ln), ln.ctypes.data, len(pt), pt.ctypes.data, pid.ctypes.data, kept.ctypes.data,
                                     off.ctypes.data, po.ctypes.data, do.ctypes.data, cap, C.byref(n)))
    idx = np.nonzero(kept)[0]
    return idx, [{int(po[k]): float(do[k]) for k in range(off[i], off[i + 1])} for i in range(len(idx))]


def op_line_match(pol_last, lines_last, pol_new, lines_new) -> Dict[int, int]:
    """TrackLSD::LineMatch through the library's host implementation: pol_* are lists of point-id collections per line."""
    def csr(pol):
        off = np.zeros(len(pol) + 1, np.int32)
        off[1:] = np.cumsum([len(p) for p in pol])
        ids = np.array([int(k) for p in pol for k in sorted(p)], np.int32)
        return off, ids
    lo, lp = csr(pol_last)
    no, npid = csr(pol_new)
    ll = np.ascontiguousarray(lines_last, np.float32).reshape(-1, 4)
    ln = np.ascontiguousarray(lines_new, np.float32).reshape(-1, 4)
    out = np.full(len(pol_new), -1, np.int32)
    L = lib()
    L.plviwo_op_line_match.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p]
    _check(L.plviwo_op_line_match(len(pol_last), lo.ctypes.data, lp.ctypes.data, ll.ctypes.data, len(pol_new), no.ctypes.data,
                                  npid.ctypes.data, ln.ctypes.data, out.ctypes.data))
    return {i: int(j) for i, j in enumerate(out) if j >= 0}


def op_ransac_fundamental(p0n, p1n, threshold: float, confidence: float = 0.999):
    """Host-side sequential step (no GPU needed): returns (mask uint8, n_inliers or -1 when OpenCV returns no mask)."""
    a = np.ascontiguousarray(p0n, np.float32).reshape(-1, 2)
    b = np.ascontiguousarray(p1n, np.float32).reshape(-1, 2)
    mask = np.zeros((len(a),), np.uint8)
    n = C.c_int(0)
    _check(lib().plviwo_op_ransac_fundamental(a.ctypes.data, b.ctypes.data, len(a), threshold, confidence, mask.ctypes.data,
                                              C.byref(n)))
    return mask, n.value
