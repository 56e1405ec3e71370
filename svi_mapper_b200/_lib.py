"""ctypes binding of libsvi_gpu.so (include/svi_gpu.h).  Fails loudly when the library is
missing or cannot be loaded -- there is no Python/CPU fallback for any entry point."""
from __future__ import annotations

import ctypes as C
import pathlib

import os

# SVI_GPU_LIB selects an alternate build of the same library (kernel tuning experiments)
LIB_PATH = pathlib.Path(os.environ.get("SVI_GPU_LIB") or (pathlib.Path(__file__).resolve().parent / "libsvi_gpu.so"))

SVI_SUCCESS = 0
SVI_ERR_INVALID, SVI_ERR_CUDA, SVI_ERR_CAPACITY, SVI_ERR_NO_DEVICE, SVI_ERR_UNSUPPORTED = -1, -2, -3, -4, -5

# svi_status
(SVI_OK, SVI_TRI_RANGE, SVI_TRI_NO_DESC, SVI_TRI_NO_MATCH, SVI_TRI_DISTANCE, SVI_TRI_ZERO_DISP, SVI_TRI_BAD_ROI,
 SVI_TRK_DEPTH, SVI_TRK_STAGE1_DIST, SVI_TRK_TRI_DESC, SVI_TRK_OUT_OF_FOV, SVI_TRK_NO_FEATURES, SVI_TRK_NO_MATCHES,
 SVI_TRK_DESC, SVI_TRK_RANGE, SVI_EPI_OUT_OF_SIGHT, SVI_EPI_VERTICAL, SVI_EPI_NEG_SLOPE, SVI_EPI_POS_SLOPE, SVI_EPI_ZERO_LEN,
 SVI_EPI_POOL_EMPTY, SVI_EPI_NO_MATCHES, SVI_EPI_DIST, SVI_EPI_ORIG_DIST, SVI_EPI_NO_TRANSLATION) = range(25)

EXPORTS = (
    "svi_params_default", "svi_status_text", "svi_brief_table_info", "svi_create", "svi_destroy", "svi_last_error", "svi_device_count",
    "svi_stereo_frames", "svi_stereo_frames_device", "svi_check_overflow", "svi_mask_active_landmarks", "svi_stereo_frame_masked", "svi_harris_response", "svi_detect", "svi_describe",
    "svi_match_hamming", "svi_match_epipolar", "svi_triangulate_right", "svi_triangulate_left", "svi_point_in_left",
    "svi_track_landmarks", "svi_track_landmarks_stages", "svi_set_profiling", "svi_stage_timings", "svi_config", "svi_kernels_per_chunk", "svi_optimize_landmarks",
    "svi_solve_stereo_posit", "svi_track_frame_stereo_only",
    "svi_multi_create", "svi_multi_destroy", "svi_multi_last_error", "svi_multi_device_count", "svi_multi_frame_range",
    "svi_multi_stereo_frames", "svi_rectify_map", "svi_set_rectification", "svi_rectify", "svi_multi_set_rectification",
)

u8p, i32p, f32p, f64p = C.POINTER(C.c_uint8), C.POINTER(C.c_int32), C.POINTER(C.c_float), C.POINTER(C.c_double)


class Camera(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("P", C.c_double * 12)]


class Params(C.Structure):
    _fields_ = [
        ("quality_level", C.c_double), ("min_distance", C.c_double), ("harris_k", C.c_double),
        ("min_disparity_px", C.c_double),
        ("max_corners", C.c_int32), ("keypoint_size", C.c_float), ("search_range_px", C.c_float),
        ("match_cutoff", C.c_float), ("cutoff_stage1", C.c_float), ("cutoff_stage2", C.c_float),
        ("cutoff_stage3", C.c_float), ("cutoff_original", C.c_float),
        ("max_candidates", C.c_int32), ("chunk_frames", C.c_int32), ("max_queries", C.c_int32),
        ("detector", C.c_int32), ("fast_threshold", C.c_int32), ("fast_nonmax", C.c_int32),
    ]


class StereoResult(C.Structure):
    _fields_ = [
        ("capacity_per_frame", C.c_int32), ("n_keypoints", C.c_void_p), ("n_detected", C.c_void_p),
        ("uv_left", C.c_void_p), ("uv_right", C.c_void_p), ("xyz_left", C.c_void_p),
        ("desc_left", C.c_void_p), ("desc_right", C.c_void_p), ("distance", C.c_void_p),
        ("match_index", C.c_void_p), ("status", C.c_void_p),
    ]


class TriResult(C.Structure):
    _fields_ = [("uv", C.c_void_p), ("xyz_left", C.c_void_p), ("desc", C.c_void_p), ("distance", C.c_void_p),
                ("match_index", C.c_void_p), ("status", C.c_void_p)]


class Landmarks(C.Structure):
    _fields_ = [("xyz_world", C.c_void_p), ("last_desc_left", C.c_void_p), ("last_desc_right", C.c_void_p),
                ("last_disparity", C.c_void_p), ("keypoint_size", C.c_void_p), ("uv_reference_left", C.c_void_p),
                ("desc_reference_left", C.c_void_p), ("T_left_to_world_at_detection", C.c_void_p)]


class TrackResult(C.Structure):
    _fields_ = [("status", C.c_void_p), ("stage", C.c_void_p), ("uv_left", C.c_void_p), ("uv_right", C.c_void_p),
                ("xyz_left", C.c_void_p), ("desc_left", C.c_void_p), ("desc_right", C.c_void_p)]


class LandmarkMeasurements(C.Structure):
    _fields_ = [("xyz_world_guess", C.c_void_p), ("first", C.c_void_p), ("pose_index", C.c_void_p), ("uv_left", C.c_void_p),
                ("uv_right", C.c_void_p), ("proj_world_to_left", C.c_void_p), ("proj_world_to_right", C.c_void_p), ("n_poses", C.c_int32)]


class OptimizeResult(C.Structure):
    _fields_ = [("xyz_world", C.c_void_p), ("outcome", C.c_void_p), ("average_squared_error", C.c_void_p), ("iterations", C.c_void_p)]


class PositProblem(C.Structure):
    """svi_posit_problem: one frame's measurements (WORLD points, LEFT / RIGHT image points) and the solver's priors."""
    _fields_ = [("n", C.c_int32), ("xyz_world", C.c_void_p), ("uv_left", C.c_void_p), ("uv_right", C.c_void_p),
                ("T_estimate", C.c_double * 16), ("T_last", C.c_double * 16), ("t_imu", C.c_double * 3)]


class PositResult(C.Structure):
    _fields_ = [("T_world_to_left", C.c_double * 16), ("outcome", C.c_uint8), ("iterations", C.c_int32), ("inliers", C.c_int32),
                ("average_squared_error", C.c_double), ("risk", C.c_double)]


class SvFrame(C.Structure):
    """svi_sv_frame: the active landmarks, their flags and the priors of one stereo-only tracking frame."""
    _fields_ = [("landmarks", Landmarks), ("flags", C.c_void_p), ("T_estimate", C.c_double * 16), ("T_estimate_damped", C.c_double * 16),
                ("T_last", C.c_double * 16), ("t_imu", C.c_double * 3), ("motion_scaling", C.c_double)]


class SvFrameResult(C.Structure):
    _fields_ = [("T_world_to_left", C.c_double * 16), ("source", C.c_uint8), ("attempts", C.c_int32), ("attempt", PositResult * 2), ("measurements", C.c_int32 * 2),
                ("pose_stage", TrackResult), ("route", C.c_void_p), ("epipolar_stage", TrackResult)]


class Rectification(C.Structure):
    """svi_rectification: matIntrinsic, vecDistortionCoefficients (k1 k2 p1 p2), matRectification, map type."""
    _fields_ = [("K", C.c_double * 9), ("D", C.c_double * 4), ("R", C.c_double * 9), ("float_maps", C.c_int32)]


(SVI_OPT_SKIPPED, SVI_OPT_CONVERGED, SVI_OPT_OPTIMAL, SVI_OPT_REJECTED, SVI_OPT_NOT_CONVERGED) = range(5)
(SVI_POSIT_OK, SVI_POSIT_TOO_FEW_POINTS, SVI_POSIT_INACCURATE, SVI_POSIT_HIGH_RISK, SVI_POSIT_NOT_CONVERGED) = range(5)
SVI_SV_POSE_CANDIDATE, SVI_SV_LEAVES = 1, 2
(SVI_SV_POSIT, SVI_SV_POSIT_DAMPED, SVI_SV_PRIOR) = range(3)
(SVI_SV_ROUTE_POSE, SVI_SV_ROUTE_EPIPOLAR, SVI_SV_ROUTE_REGIONAL, SVI_SV_ROUTE_REGIONAL_NO_TRANSLATION, SVI_SV_ROUTE_DROPPED) = range(1, 6)

_lib = None
_others: dict = {}


def load(path=None):
    """Load libsvi_gpu.so once; raise with a build hint if it is absent.  `path` loads another build of the same
    library (a variant compiled around a different BRIEF pair table, a tuning experiment) beside the default one."""
    global _lib
    if path is None and _lib is not None:
        return _lib
    if path is not None and str(path) in _others:
        return _others[str(path)]
    lib_path = pathlib.Path(path) if path is not None else LIB_PATH
    if not lib_path.exists():
        raise ImportError(
            f"{lib_path} is missing: build it with `python -m svi_mapper_b200.build` "
            "(svi_mapper_b200 has no CPU fallback)")
    lib = C.CDLL(str(lib_path))
    vp, sz, ci = C.c_void_p, C.c_size_t, C.c_int
    lib.svi_params_default.argtypes = [C.POINTER(Params)]
    lib.svi_status_text.argtypes = [ci]
    lib.svi_status_text.restype = C.c_char_p
    lib.svi_brief_table_info.argtypes = []
    lib.svi_brief_table_info.restype = C.c_char_p
    lib.svi_create.argtypes = [C.POINTER(Camera), C.POINTER(Camera), C.POINTER(Params), ci, C.POINTER(vp)]
    lib.svi_destroy.argtypes = [vp]
    lib.svi_destroy.restype = None
    lib.svi_last_error.argtypes = [vp]
    lib.svi_last_error.restype = C.c_char_p
    lib.svi_device_count.argtypes = []
    lib.svi_stereo_frames.argtypes = [vp, vp, vp, sz, sz, ci, vp, C.POINTER(StereoResult)]
    lib.svi_stereo_frames_device.argtypes = [vp, vp, vp, sz, sz, ci, vp, C.POINTER(StereoResult), vp]
    lib.svi_check_overflow.argtypes = [vp]
    lib.svi_mask_active_landmarks.argtypes = [vp, vp, ci, vp, sz]
    lib.svi_stereo_frame_masked.argtypes = [vp, vp, vp, sz, vp, ci, C.POINTER(StereoResult)]
    lib.svi_harris_response.argtypes = [vp, vp, sz, vp]
    lib.svi_detect.argtypes = [vp, vp, sz, sz, ci, vp, vp, vp]
    lib.svi_describe.argtypes = [vp, vp, sz, vp, ci, vp, vp]
    lib.svi_match_hamming.argtypes = [vp, vp, ci, vp, ci, vp, vp]
    lib.svi_match_epipolar.argtypes = [vp, vp, vp, ci, vp, vp, ci, C.c_float, C.c_float, C.c_float, vp, vp, vp]
    lib.svi_triangulate_right.argtypes = [vp, vp, sz, ci, vp, vp, vp, C.c_float, C.POINTER(TriResult)]
    lib.svi_triangulate_left.argtypes = [vp, vp, sz, ci, vp, vp, vp, vp, C.c_float, C.POINTER(TriResult)]
    lib.svi_point_in_left.argtypes = [vp, ci, vp, vp, vp, vp]
    lib.svi_track_landmarks.argtypes = [vp, vp, vp, sz, vp, C.POINTER(Landmarks), ci, C.c_double, C.POINTER(TrackResult)]
    lib.svi_track_landmarks_stages.argtypes = [vp, vp, vp, sz, vp, C.POINTER(Landmarks), ci, C.c_double, C.c_uint32, C.POINTER(TrackResult)]
    lib.svi_set_profiling.argtypes = [vp, ci]
    lib.svi_stage_timings.argtypes = [vp, C.POINTER(C.c_char_p), f64p, C.POINTER(C.c_int64), ci]
    lib.svi_config.argtypes = [vp, i32p, i32p, i32p]
    lib.svi_kernels_per_chunk.argtypes = [vp, ci]
    lib.svi_optimize_landmarks.argtypes = [vp, C.POINTER(LandmarkMeasurements), ci, C.POINTER(OptimizeResult)]
    lib.svi_solve_stereo_posit.argtypes = [vp, C.POINTER(PositProblem), C.POINTER(PositResult)]
    lib.svi_track_frame_stereo_only.argtypes = [vp, vp, vp, sz, C.POINTER(SvFrame), ci, C.POINTER(SvFrameResult)]
    lib.svi_multi_create.argtypes = [C.POINTER(Camera), C.POINTER(Camera), C.POINTER(Params), i32p, ci, C.POINTER(vp)]
    lib.svi_multi_destroy.argtypes = [vp]
    lib.svi_multi_destroy.restype = None
    lib.svi_multi_last_error.argtypes = [vp]
    lib.svi_multi_last_error.restype = C.c_char_p
    lib.svi_multi_device_count.argtypes = [vp]
    lib.svi_multi_frame_range.argtypes = [vp, ci, ci, i32p, i32p]
    lib.svi_multi_stereo_frames.argtypes = [vp, vp, vp, sz, sz, ci, vp, C.POINTER(StereoResult)]
    lib.svi_rectify_map.argtypes = [C.POINTER(Camera), C.POINTER(Rectification), vp, vp]
    lib.svi_set_rectification.argtypes = [vp, C.POINTER(Rectification), C.POINTER(Rectification)]
    lib.svi_rectify.argtypes = [vp, ci, vp, sz, sz, ci, vp, sz]
    lib.svi_multi_set_rectification.argtypes = [vp, C.POINTER(Rectification), C.POINTER(Rectification)]
    for name in EXPORTS:
        getattr(lib, name)  # AttributeError here = header/library mismatch
    if path is None:
        _lib = lib
    else:
        _others[str(path)] = lib
    return lib
