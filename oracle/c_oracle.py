"""ctypes wrapper of oracle/svi_oracle.c (TEST INFRASTRUCTURE / CPU baseline only)."""
from __future__ import annotations

import ctypes as C
import os
import pathlib
import subprocess

import numpy as np

HERE = pathlib.Path(__file__).resolve().parent


class Config(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("P_left", C.c_double * 12), ("P_right", C.c_double * 12),
                ("quality_level", C.c_double), ("min_distance", C.c_double), ("harris_k", C.c_double),
                ("min_disparity", C.c_double), ("max_corners", C.c_int32), ("keypoint_size", C.c_float),
                ("search_range", C.c_float), ("match_cutoff", C.c_float)]


class Result(C.Structure):
    _fields_ = [("capacity", C.c_int32), ("uv_left", C.c_void_p), ("uv_right", C.c_void_p), ("xyz_left", C.c_void_p),
                ("desc_left", C.c_void_p), ("desc_right", C.c_void_p), ("distance", C.c_void_p),
                ("match_index", C.c_void_p), ("status", C.c_void_p)]


class TrackParams(C.Structure):
    _fields_ = [("cutoff_stage1", C.c_float), ("cutoff_stage2", C.c_float), ("cutoff_stage3", C.c_float), ("cutoff_original", C.c_float),
                ("epipolar_base_length", C.c_double), ("block_size_stage2", C.c_int32)]


class Landmarks(C.Structure):
    _fields_ = [("xyz_world", C.c_void_p), ("last_desc_left", C.c_void_p), ("last_desc_right", C.c_void_p), ("last_disparity", C.c_void_p),
                ("keypoint_size", C.c_void_p), ("uv_reference_left", C.c_void_p), ("desc_reference_left", C.c_void_p),
                ("T_left_to_world_at_detection", C.c_void_p)]


class TrackResult(C.Structure):
    _fields_ = [("status", C.c_void_p), ("stage", C.c_void_p), ("uv_left", C.c_void_p), ("uv_right", C.c_void_p), ("xyz_left", C.c_void_p),
                ("desc_left", C.c_void_p), ("desc_right", C.c_void_p)]


def build(native: bool = False, out: pathlib.Path | None = None) -> pathlib.Path:
    """make the portable or the -march=native library; `out` is where the native one goes instead of oracle/."""
    target = HERE / ("libsvi_oracle_native.so" if native else "libsvi_oracle.so")
    cmd = ["make", "-C", str(HERE), "native" if native else "all"]
    if native and out is not None:
        target = pathlib.Path(out).resolve()
        cmd.append(f"NATIVE={target}")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + r.stdout + r.stderr)
    return target


def build_variant(pattern_header: pathlib.Path, out: pathlib.Path) -> pathlib.Path:
    """The checker compiled around another BRIEF pair table (header from tools/gen_pattern_header.py --table)."""
    out = pathlib.Path(out)
    src = HERE / "svi_oracle.c"
    if out.exists() and out.stat().st_mtime >= max(src.stat().st_mtime, pathlib.Path(pattern_header).stat().st_mtime):
        return out
    cmd = ["gcc", "-O3", "-std=gnu11", "-fPIC", "-ffp-contract=off", "-march=x86-64-v3", f'-DSVI_BRIEF_PATTERN_HEADER="{pattern_header}"',
           "-shared", "-o", str(out), str(src), "-lm", "-lpthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("oracle variant build failed:\n" + r.stdout + r.stderr)
    return out


_libs: dict = {}


def load(native=False):
    """Load (building if needed and possible) the oracle library.  `native` may also be the path of a variant built
    around another BRIEF pair table (svi_mapper_b200.build.build_with_table)."""
    key = native if isinstance(native, bool) else str(native)
    if key in _libs:
        return _libs[key]
    if isinstance(native, bool):
        path = HERE / ("libsvi_oracle_native.so" if native else "libsvi_oracle.so")
        src = HERE / "svi_oracle.c"
        if not path.exists() or path.stat().st_mtime < src.stat().st_mtime:
            path = build(native)
    else:
        path = pathlib.Path(native)
    lib = C.CDLL(str(path))
    vp, ci, cf = C.c_void_p, C.c_int, C.c_float
    lib.svo_harris_response.argtypes = [vp, ci, ci, ci, C.c_double, vp]
    lib.svo_gftt.argtypes = [vp, ci, ci, ci, vp, ci, ci, C.c_double, C.c_double, C.c_double, vp, ci]
    lib.svo_brief32.argtypes = [vp, ci, ci, ci, vp, ci, vp, vp]
    lib.svo_match.argtypes = [vp, vp, ci, vp]
    lib.svo_point_in_left.argtypes = [C.POINTER(Config), vp, vp, vp]
    lib.svo_triangulate_right.argtypes = [C.POINTER(Config), vp, ci, cf, cf, cf, vp, vp, vp, vp, vp, vp, vp]
    lib.svo_triangulate_left.argtypes = [C.POINTER(Config), vp, ci, cf, cf, cf, cf, vp, vp, vp, vp, vp, vp, vp]
    lib.svo_stereo_frames_mt.argtypes = [C.POINTER(Config), vp, vp, ci, C.c_size_t, ci, vp, C.POINTER(Result), vp, vp, ci]
    lib.svo_harris_response_roi.argtypes = [vp, ci, ci, ci, ci, ci, ci, ci, C.c_double, vp]
    lib.svo_gftt_roi.argtypes = [vp, ci, ci, ci, ci, ci, ci, ci, ci, C.c_double, C.c_double, C.c_double, vp, ci]
    lib.svo_track_params_default.argtypes = [C.POINTER(TrackParams)]
    lib.svo_optimize_landmark.argtypes = [vp, ci, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.svo_solve_stereo_posit.argtypes = [vp, vp, vp, vp, vp, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.svo_track_landmarks.argtypes = [C.POINTER(Config), C.POINTER(TrackParams), vp, vp, ci, vp, C.POINTER(Landmarks), ci, C.c_double,
                                        C.c_uint, C.POINTER(TrackResult), ci]
    _libs[key] = lib
    return lib


def make_config(cam_left, cam_right, max_corners=1000, quality_level=0.01, min_distance=7.0, harris_k=0.04,
                min_disparity=0.01, keypoint_size=7.0, search_range=60.0, match_cutoff=100.0) -> Config:
    c = Config()
    c.width, c.height = int(cam_left.width), int(cam_left.height)
    pl, pr = np.asarray(cam_left.P, np.float64).reshape(12), np.asarray(cam_right.P, np.float64).reshape(12)
    for i in range(12):
        c.P_left[i], c.P_right[i] = float(pl[i]), float(pr[i])
    c.quality_level, c.min_distance, c.harris_k, c.min_disparity = quality_level, min_distance, harris_k, min_disparity
    c.max_corners, c.keypoint_size, c.search_range, c.match_cutoff = max_corners, keypoint_size, search_range, match_cutoff
    return c


def harris_response(img: np.ndarray, k=0.04, native=False) -> np.ndarray:
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    out = np.empty((h, w), np.float32)
    rc = load(native).svo_harris_response(img.ctypes.data, w, h, w, k, out.ctypes.data)
    assert rc == 0
    return out


def gftt(img: np.ndarray, max_corners=1000, quality=0.01, min_distance=7.0, mask=None, k=0.04, native=False) -> np.ndarray:
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    cap = max_corners if max_corners > 0 else w * h // 4
    xy = np.zeros((cap, 2), np.int32)
    m = np.ascontiguousarray(mask, np.uint8) if mask is not None else None
    n = load(native).svo_gftt(img.ctypes.data, w, h, w, m.ctypes.data if m is not None else None, w, max_corners, quality,
                              min_distance, k, xy.ctypes.data, cap)
    assert n >= 0
    return xy[:n].copy()


def brief32(img: np.ndarray, pts, native=False):
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    p = np.ascontiguousarray(np.asarray(pts, np.float32).reshape(-1, 2))
    n = len(p)
    desc = np.zeros((max(n, 1), 32), np.uint8)
    kept = np.zeros(max(n, 1), np.int32)
    nk = load(native).svo_brief32(img.ctypes.data, w, h, w, p.ctypes.data, n, desc.ctypes.data, kept.ctypes.data)
    assert nk >= 0
    return kept[:nk].copy(), desc[:nk].copy()


def stereo_frames(cfg: Config, left: np.ndarray, right: np.ndarray, masks=None, n_threads: int = 1, native=False) -> dict:
    """svo_stereo_frames_mt on (n, H, W) uint8 batches -> dict of (n, cap, ...) arrays + counts."""
    L = np.ascontiguousarray(left, np.uint8)
    R = np.ascontiguousarray(right, np.uint8)
    if L.ndim == 2:
        L, R = L[None], R[None]
    n, h, w = L.shape
    cap = int(cfg.max_corners)
    M = np.ascontiguousarray(masks, np.uint8).reshape(n, h, w) if masks is not None else None
    out = dict(uv_left=np.zeros((n, cap, 2), np.float32), uv_right=np.zeros((n, cap, 2), np.float32),
               xyz_left=np.zeros((n, cap, 3), np.float64), desc_left=np.zeros((n, cap, 32), np.uint8),
               desc_right=np.zeros((n, cap, 32), np.uint8), distance=np.full((n, cap), -1, np.int32),
               match_index=np.full((n, cap), -1, np.int32), status=np.zeros((n, cap), np.uint8),
               n_keypoints=np.zeros(n, np.int32), n_detected=np.zeros(n, np.int32))
    r = Result(cap, out["uv_left"].ctypes.data, out["uv_right"].ctypes.data, out["xyz_left"].ctypes.data,
               out["desc_left"].ctypes.data, out["desc_right"].ctypes.data, out["distance"].ctypes.data,
               out["match_index"].ctypes.data, out["status"].ctypes.data)
    rc = load(native).svo_stereo_frames_mt(C.byref(cfg), L.ctypes.data, R.ctypes.data, w, w * h, n,
                                           M.ctypes.data if M is not None else None, C.byref(r),
                                           out["n_keypoints"].ctypes.data, out["n_detected"].ctypes.data, int(n_threads))
    assert rc == 0
    return out


def track_landmarks(cfg: Config, img_left, img_right, T_world_to_left, xyz_world, last_desc_left, last_desc_right, last_disparity,
                    keypoint_size, motion_scaling: float, uv_reference_left=None, desc_reference_left=None,
                    T_left_to_world_at_detection=None, stages=None, n_threads: int = 1, native=False, **cutoffs) -> dict:
    """svo_track_landmarks: CFundamentalMatcher::trackManual (all stages) for n landmarks of one pair; the same arguments
    and result keys as StereoFrontend.track_landmarks.  cutoffs: cutoff_stage1 / 2 / 3 / cutoff_original overrides."""
    lib = load(native)
    a = np.ascontiguousarray(img_left, np.uint8)
    b = np.ascontiguousarray(img_right, np.uint8)
    h, w = a.shape
    T = np.ascontiguousarray(np.asarray(T_world_to_left, np.float64).reshape(4, 4))
    xw = np.ascontiguousarray(np.asarray(xyz_world, np.float64).reshape(-1, 3))
    n = len(xw)
    dl = np.ascontiguousarray(np.asarray(last_desc_left, np.uint8).reshape(n, 32))
    dr = np.ascontiguousarray(np.asarray(last_desc_right, np.uint8).reshape(n, 32))
    disp = np.ascontiguousarray(np.asarray(last_disparity, np.float32).reshape(n))
    size = np.ascontiguousarray(np.broadcast_to(np.asarray(keypoint_size, np.float32), (n,)).copy())
    uvref = dref = tdet = None
    if uv_reference_left is not None:
        uvref = np.ascontiguousarray(np.asarray(uv_reference_left, np.float64).reshape(n, 2))
        dref = np.ascontiguousarray(np.asarray(desc_reference_left, np.uint8).reshape(n, 32))
        tdet = np.ascontiguousarray(np.broadcast_to(np.asarray(T_left_to_world_at_detection, np.float64), (n, 4, 4)).copy())
    if stages is None:
        stages = 3 | (4 if uvref is not None else 0)
    out = dict(status=np.zeros(n, np.uint8), stage=np.zeros(n, np.uint8), uv_l=np.zeros((n, 2), np.float32),
               uv_r=np.zeros((n, 2), np.float32), xyz=np.zeros((n, 3), np.float64), desc_l=np.zeros((n, 32), np.uint8),
               desc_r=np.zeros((n, 32), np.uint8))
    p = lambda x: x.ctypes.data if x is not None else None
    lm = Landmarks(p(xw), p(dl), p(dr), p(disp), p(size), p(uvref), p(dref), p(tdet))
    r = TrackResult(p(out["status"]), p(out["stage"]), p(out["uv_l"]), p(out["uv_r"]), p(out["xyz"]), p(out["desc_l"]), p(out["desc_r"]))
    tp = TrackParams()
    lib.svo_track_params_default(C.byref(tp))
    for k, v in cutoffs.items():
        setattr(tp, k, v)
    rc = lib.svo_track_landmarks(C.byref(cfg), C.byref(tp), a.ctypes.data, b.ctypes.data, w, T.ctypes.data, C.byref(lm), n,
                                 float(motion_scaling), int(stages), C.byref(r), int(n_threads))
    assert rc == 0
    return out


def frame(out: dict, f: int) -> dict:
    n = int(out["n_keypoints"][f])
    return dict(uv_l=out["uv_left"][f, :n], uv_r=out["uv_right"][f, :n], xyz=out["xyz_left"][f, :n],
                desc_l=out["desc_left"][f, :n], desc_r=out["desc_right"][f, :n], dist=out["distance"][f, :n],
                idx=out["match_index"][f, :n], status=out["status"][f, :n])


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def optimize_landmark(xyz_guess, measurements, native=False) -> dict:
    """svo_optimize_landmark: CLandmark::optimize for one landmark; measurements = list of (P_world_to_left 3x4,
    P_world_to_right 3x4, uv_left, uv_right) like oracle.frontend_np.optimize_landmark.  Returns dict(xyz, outcome,
    average_squared_error, iterations) with outcome 0 skipped / 1 converged / 2 optimal / 3 rejected / 4 not converged."""
    m = len(measurements)
    g = np.ascontiguousarray(np.asarray(xyz_guess, np.float64).reshape(3))
    pl = np.ascontiguousarray(np.stack([np.asarray(q[0], np.float64).reshape(12) for q in measurements])) if m else np.zeros((0, 12))
    pr = np.ascontiguousarray(np.stack([np.asarray(q[1], np.float64).reshape(12) for q in measurements])) if m else np.zeros((0, 12))
    ul = np.ascontiguousarray(np.stack([np.asarray(q[2], np.float32).reshape(2) for q in measurements])) if m else np.zeros((0, 2), np.float32)
    ur = np.ascontiguousarray(np.stack([np.asarray(q[3], np.float32).reshape(2) for q in measurements])) if m else np.zeros((0, 2), np.float32)
    xyz = np.zeros(3, np.float64)
    outcome, iters = np.zeros(1, np.int32), np.zeros(1, np.int32)
    avg = np.zeros(1, np.float64)
    rc = load(native).svo_optimize_landmark(g.ctypes.data, m, pl.ctypes.data, pr.ctypes.data, ul.ctypes.data, ur.ctypes.data, xyz.ctypes.data,
                                            outcome.ctypes.data, avg.ctypes.data, iters.ctypes.data)
    assert rc == 0
    return dict(xyz=xyz, outcome=int(outcome[0]), average_squared_error=float(avg[0]), iterations=int(iters[0]))


def solve_stereo_posit(P_left, P_right, xyz_world, uv_left, uv_right, T_estimate, T_last=None, t_imu=None, native=False) -> dict:
    """svo_solve_stereo_posit: CSolverStereoPosit::getTransformationWORLDtoLEFT for one frame's measurements (xyz_world (n, 3)
    float64, uv_left / uv_right (n, 2) float32) from the prior T_estimate; the same arguments (plus the two 3 x 4 projection
    matrices) and result keys as StereoFrontend.solve_stereo_posit, minus `reason`.  T_last defaults to T_estimate, t_imu to zero."""
    P = [np.ascontiguousarray(np.asarray(m, np.float64).reshape(12)) for m in (P_left, P_right)]
    xw = np.ascontiguousarray(np.asarray(xyz_world, np.float64).reshape(-1, 3))
    n = len(xw)
    ul = np.ascontiguousarray(np.asarray(uv_left, np.float32).reshape(n, 2))
    ur = np.ascontiguousarray(np.asarray(uv_right, np.float32).reshape(n, 2))
    Te = np.ascontiguousarray(np.asarray(T_estimate, np.float64).reshape(16))
    Tl = Te if T_last is None else np.ascontiguousarray(np.asarray(T_last, np.float64).reshape(16))
    ti = np.zeros(3) if t_imu is None else np.ascontiguousarray(np.asarray(t_imu, np.float64).reshape(3))
    T = np.zeros(16, np.float64)
    outcome, iters, inliers = np.zeros(1, np.int32), np.zeros(1, np.int32), np.zeros(1, np.int32)
    avg, risk = np.zeros(1, np.float64), np.zeros(1, np.float64)
    rc = load(native).svo_solve_stereo_posit(P[0].ctypes.data, P[1].ctypes.data, Te.ctypes.data, Tl.ctypes.data, ti.ctypes.data, n, xw.ctypes.data,
                                             ul.ctypes.data, ur.ctypes.data, T.ctypes.data, outcome.ctypes.data, iters.ctypes.data,
                                             inliers.ctypes.data, avg.ctypes.data, risk.ctypes.data)
    assert rc == 0
    return dict(T=T.reshape(4, 4), outcome=int(outcome[0]), iterations=int(iters[0]), inliers=int(inliers[0]),
                average_squared_error=float(avg[0]), risk=float(risk[0]))
