"""One frame of the stereo-only tracker in one call (svi_track_frame_stereo_only): against the composed calls it replaces
(track_landmarks on stage subsets, solve_stereo_posit, the damped retry, the epipolar / regional split), on raw frames with
rectification set, and through the C++ tracker CTrackerSV (facade_demo --sequence-sv) against its composed CPU-solve path."""
import ctypes as C
import os
import pathlib
import subprocess
import sys

import numpy as np
import pytest

from svi_mapper_b200 import StereoFrontend, _lib

ROOT = pathlib.Path(__file__).resolve().parents[1]
CALIB = ROOT / "tests" / "golden" / "calib"
EXE = ROOT / "svi_mapper_b200" / "host" / "facade_demo"

pytestmark = pytest.mark.usefixtures("built_library")

TRACK_KEYS = ("status", "stage", "uv_l", "uv_r", "xyz", "desc_l", "desc_r")


def _cams():
    from svi_mapper_b200 import load_camera
    return load_camera(str(CALIB / "vi_sensor_left.txt")), load_camera(str(CALIB / "vi_sensor_right.txt"))


def test_track_frame_stereo_only_refuses_a_null_context():
    lib = _lib.load()
    fr, res = _lib.SvFrame(), _lib.SvFrameResult()
    img = np.zeros(64, np.uint8)
    assert lib.svi_track_frame_stereo_only(None, img.ctypes.data, img.ctypes.data, 8, C.byref(fr), 0, C.byref(res)) == _lib.SVI_ERR_INVALID
    assert lib.svi_track_frame_stereo_only(None, None, None, 0, None, 0, None) == _lib.SVI_ERR_INVALID


@pytest.mark.gpu
def test_track_frame_stereo_only_refuses_null_arrays():
    """With a context and n > 0, a null input or output array is refused before any work, as are unknown flag bits."""
    cams = _cams()
    n, W, H = 4, cams[0].width, cams[0].height
    img = np.zeros((H, W), np.uint8)
    keep = []

    def arr(shape, dt):
        a = np.zeros(shape, dt)
        keep.append(a)
        return a.ctypes.data

    def frame():
        fr = _lib.SvFrame(_lib.Landmarks(arr((n, 3), np.float64), arr((n, 32), np.uint8), arr((n, 32), np.uint8), arr(n, np.float32), arr(n, np.float32),
                                         arr((n, 2), np.float64), arr((n, 32), np.uint8), arr((n, 16), np.float64)), arr(n, np.uint8))
        fr.motion_scaling = 1.0
        return fr

    def track():
        return _lib.TrackResult(arr(n, np.uint8), arr(n, np.uint8), arr((n, 2), np.float32), arr((n, 2), np.float32), arr((n, 3), np.float64),
                                arr((n, 32), np.uint8), arr((n, 32), np.uint8))

    with StereoFrontend(*cams) as fe:
        lib = fe._lib

        def call(fr, res):
            return lib.svi_track_frame_stereo_only(fe._ctx, img.ctypes.data, img.ctypes.data, W, C.byref(fr), n, C.byref(res))
        for field in ("flags", "landmarks.T_left_to_world_at_detection", "landmarks.xyz_world", "route", "pose_stage.desc_right",
                      "epipolar_stage.status"):
            fr, res = frame(), _lib.SvFrameResult(pose_stage=track(), route=arr(n, np.uint8), epipolar_stage=track())
            obj, name = (fr, field) if field in ("flags",) or field.startswith("landmarks") else (res, field)
            if "." in name:
                head, name = name.split(".")
                obj = getattr(obj, head)
            setattr(obj, name, None)
            assert call(fr, res) == _lib.SVI_ERR_INVALID, field
            assert b"null array" in lib.svi_last_error(fe._ctx), field
        fr, res = frame(), _lib.SvFrameResult(pose_stage=track(), route=arr(n, np.uint8), epipolar_stage=track())
        flags = np.full(n, 4, np.uint8)
        fr.flags = flags.ctypes.data
        assert call(fr, res) == _lib.SVI_ERR_INVALID


# ----------------------------------------------------------------------------------------------------------- the reference
def _host_translation_moved(T, T_det):
    """trackEpipolar's verdict (CFundamentalMatcher.h:561-563) in the host's arithmetic, element by element: the translation
    column of Isometry3d::operator*(T, T_det) (host/Types.h:125, the sum starting at 0.0), then its squared norm > 0."""
    t = []
    for r in range(3):
        s = np.zeros(len(T_det))
        for k in range(3):
            s = s + T[r, k] * T_det[:, k, 3]
        t.append(s + T[r, 3])
    return 0.0 < (t[0] * t[0] + t[1] * t[1]) + t[2] * t[2]


def _subset(st, idx):
    return {k: v[idx] for k, v in st.items()}


def _track(fe, L, R, T, st, scaling, stages, with_reference):
    ref = dict(uv_reference_left=st["uv_ref"], desc_reference_left=st["ref_desc_l"], T_left_to_world_at_detection=st["T_det"]) if with_reference else {}
    return fe.track_landmarks(L, R, T, st["xyz_w"], st["last_desc_l"], st["last_desc_r"], st["last_disp"], 7.0, scaling, stages=stages, **ref)


def composed(fe, L, R, st, flags, T_est, T_damped, T_last, t_imu, scaling):
    """What CTrackerSV::process does today through the separate calls: getPoseStereoPosit with its damped retry, then trackEpipolar."""
    n = len(flags)
    zeros = lambda: {k: np.zeros((n,) + v.shape[1:], v.dtype) for k, v in fe._track_out(0)[0].items()}
    pose, epi = zeros(), zeros()
    cand = np.flatnonzero(flags & 1)
    attempts, measurements, accepted = [], [], None
    for a, T_prior in enumerate((T_est, T_damped)):
        r = _track(fe, L, R, T_prior, _subset(st, cand), scaling, 3, False)
        hit = r["stage"] > 0
        measurements.append(int(hit.sum()))
        attempts.append(fe.solve_stereo_posit(st["xyz_w"][cand][hit], r["uv_l"][hit], r["uv_r"][hit], T_prior, T_last, t_imu))
        for k in TRACK_KEYS:
            pose[k][cand] = r[k]
        if attempts[-1]["outcome"] == _lib.SVI_POSIT_OK:
            accepted = a
            break
    T = attempts[accepted]["T"] if accepted is not None else np.asarray(T_damped, np.float64)
    route = np.where(flags & 2, _lib.SVI_SV_ROUTE_DROPPED, 0).astype(np.uint8)
    if accepted is not None:
        route[pose["stage"] > 0] = _lib.SVI_SV_ROUTE_POSE
    rest = route == 0
    moved = _host_translation_moved(T, st["T_det"])
    route[rest & moved] = _lib.SVI_SV_ROUTE_EPIPOLAR
    route[rest & ~moved] = _lib.SVI_SV_ROUTE_REGIONAL
    e = np.flatnonzero(route == _lib.SVI_SV_ROUTE_EPIPOLAR)
    r3 = _track(fe, L, R, T, _subset(st, e), scaling, 4, True)
    for k in TRACK_KEYS:
        epi[k][e] = r3[k]
    route[e[r3["status"] == _lib.SVI_EPI_NO_TRANSLATION]] = _lib.SVI_SV_ROUTE_REGIONAL_NO_TRANSLATION
    g = np.flatnonzero((route == _lib.SVI_SV_ROUTE_REGIONAL) | (route == _lib.SVI_SV_ROUTE_REGIONAL_NO_TRANSLATION))
    r2 = _track(fe, L, R, T, _subset(st, g), scaling, 2, False)
    for k in TRACK_KEYS:
        epi[k][g] = r2[k]
    source = ("posit", "posit-damped", "prior")[2 if accepted is None else accepted]
    return dict(T=T, source=source, attempts=attempts, measurements=measurements, route=route, pose_stage=pose, epipolar_stage=epi)


def fused(fe, L, R, st, flags, T_est, T_damped, T_last, t_imu, scaling):
    return fe.track_frame_stereo_only(L, R, st["xyz_w"], st["last_desc_l"], st["last_desc_r"], st["last_disp"], 7.0, st["uv_ref"], st["ref_desc_l"],
                                      st["T_det"], flags, T_est, T_damped, T_last, t_imu, scaling)


def assert_same(got, want, name):
    assert got["source"] == want["source"], (name, got["source"], want["source"])
    assert got["T"].tobytes() == want["T"].tobytes(), name
    assert len(got["attempts"]) == len(want["attempts"]) and got["measurements"] == want["measurements"], name
    for a, b in zip(got["attempts"], want["attempts"]):
        assert a["T"].tobytes() == b["T"].tobytes() and a["outcome"] == b["outcome"], (name, a, b)
        assert (a["iterations"], a["inliers"]) == (b["iterations"], b["inliers"]), (name, a, b)
        if b["outcome"] in (_lib.SVI_POSIT_OK, _lib.SVI_POSIT_INACCURATE, _lib.SVI_POSIT_HIGH_RISK):   # computed by these outcomes
            assert a["average_squared_error"] == b["average_squared_error"], (name, a, b)
        if b["outcome"] in (_lib.SVI_POSIT_OK, _lib.SVI_POSIT_HIGH_RISK):
            assert a["risk"] == b["risk"], (name, a, b)
    assert got["route"].tobytes() == want["route"].tobytes(), name
    for part in ("pose_stage", "epipolar_stage"):
        for k in TRACK_KEYS:
            assert got[part][k].tobytes() == want[part][k].tobytes(), (name, part, k)


def _c3_state(fe, cams, frames):
    """C3 frames and the Python SequenceTracker's landmark state after tracking all but the last of them with the true poses."""
    from svi_mapper_b200.sequence import GpuBackend, SequenceTracker, render_sequence
    L, R, T = render_sequence(cams[0], cams[1], frames, 4000)
    trk = SequenceTracker(GpuBackend(fe), cams[0])
    for t in range(frames - 1):
        trk.process(L[t], R[t], T[t])
    return L, R, T, {k: v.copy() for k, v in trk.s.items()}


def _cases(fe, L, R, T, st, rng):
    """(name, L, R, state, flags, T_est, T_damped, T_last, t_imu, scaling) for every route the frame can take."""
    k = len(T) - 1
    n = len(st["uid"])
    flags = np.ones(n, np.uint8)
    mixed = rng.choice(np.array([0, 1, 2, 3], np.uint8), n, p=[0.15, 0.7, 0.1, 0.05])
    T_off = T[k].copy()
    T_off[:3, 3] += [3.0, 0.0, 0.0]
    s = 1.2
    yield "good prior", L[k], R[k], st, flags, T[k], T[k - 1], T[k - 1], np.zeros(3), s
    yield "dropped and non-candidates", L[k], R[k], st, mixed, T[k], T[k - 1], T[k - 1], np.zeros(3), s
    yield "prior 3 m off", L[k], R[k], st, flags, T_off, T[k], T[k - 1], np.zeros(3), s
    black = np.zeros_like(L[k])
    yield "black frames", black, black, st, flags, T[k], T[k - 1], T[k - 1], np.zeros(3), s
    # a pose equal to the detection pose of a third of the landmarks: no candidate, so the pose is the damped prior, which has an
    # identity rotation; those landmarks get the inverse as their detection pose, whose product with it has exactly zero translation
    T_flat = np.eye(4)
    T_flat[:3, 3] = T[k][:3, 3]
    st_reg = {kk: v.copy() for kk, v in st.items()}
    st_reg["T_det"][::3] = np.eye(4)
    st_reg["T_det"][::3, :3, 3] = -T[k][:3, 3]
    yield "regional from the start", L[k], R[k], st_reg, np.zeros(n, np.uint8), T[k], T_flat, T[k - 1], np.zeros(3), s
    empty = {kk: v[:0] for kk, v in st.items()}
    yield "n = 0", L[k], R[k], empty, np.zeros(0, np.uint8), T[k], T[k - 1], T[k - 1], np.zeros(3), s
    # exactly 25 / 26 pose hits: the stage-1/2 result of a landmark does not depend on the other landmarks of the call
    r = _track(fe, L[k], R[k], T[k], st, s, 3, False)
    hits, misses = np.flatnonzero(r["stage"] > 0), np.flatnonzero(r["stage"] == 0)
    for m in (25, 26):
        f = np.zeros(n, np.uint8)
        f[hits[:m]] = 1
        f[misses[:40]] = 1
        yield f"{m} pose hits", L[k], R[k], st, f, T[k], T[k], T[k - 1], np.zeros(3), s


@pytest.mark.gpu
def test_fused_frame_equals_the_composed_calls():
    """Every output of the fused call -- pose, source, solve attempts, route, both per-landmark results -- equals, byte for byte,
    what the composed calls give on C3 landmark states: a good prior, a prior 3 m off (the damped retry), black frames (both solves
    fail), a pose with no translation since detection (the regional route), dropped and non-candidate landmarks, n = 0 and the
    25 / 26 point boundary of the solver."""
    cams = _cams()
    rng = np.random.default_rng(7)
    with StereoFrontend(*cams, max_corners=4000) as fe:
        L, R, T, st = _c3_state(fe, cams, 9)
        assert len(st["uid"]) > 300
        sources, routes = set(), set()
        for name, *args in _cases(fe, L, R, T, st, rng):
            want = composed(fe, *args)
            got = fused(fe, *args)
            assert_same(got, want, name)
            sources.add(got["source"])
            routes.update(np.unique(got["route"]).tolist())
            if name == "prior 3 m off":
                assert got["source"] == "posit-damped" and got["attempts"][0]["outcome"] != _lib.SVI_POSIT_OK, got["attempts"]
            if name == "black frames":
                assert [a["outcome"] for a in got["attempts"]] == [_lib.SVI_POSIT_TOO_FEW_POINTS] * 2
            if name.endswith("pose hits"):
                m = int(name.split()[0])
                assert int((got["pose_stage"]["stage"] > 0).sum()) == m and got["measurements"][0] == m
                assert (got["attempts"][0]["outcome"] == _lib.SVI_POSIT_TOO_FEW_POINTS) == (m == 25)
        assert sources == {"posit", "posit-damped", "prior"}, sources
        assert {_lib.SVI_SV_ROUTE_POSE, _lib.SVI_SV_ROUTE_EPIPOLAR, _lib.SVI_SV_ROUTE_REGIONAL, _lib.SVI_SV_ROUTE_DROPPED} <= routes, routes


@pytest.mark.gpu
def test_fused_frame_on_raw_frames_with_rectification():
    """Raw frames with set_rectification give what the cv2-rectified frames give without it."""
    import cv2
    from svi_mapper_b200.synth import unrectify
    cams = _cams()

    def rect(cam, raw):   # cv2's scalar code paths on one thread, as the library's maps are pinned to them
        opt, threads = cv2.useOptimized(), cv2.getNumThreads()
        cv2.setUseOptimized(False)
        cv2.setNumThreads(1)
        try:
            m1, m2 = cv2.initUndistortRectifyMap(cam.K, cam.distortion, cam.rectification, cam.P, (cam.width, cam.height), cv2.CV_16SC2)
            return cv2.remap(raw, m1, m2, cv2.INTER_LINEAR)
        finally:
            cv2.setUseOptimized(opt)
            cv2.setNumThreads(threads)
    with StereoFrontend(*cams, max_corners=4000) as plain, StereoFrontend(*cams, max_corners=4000) as raw:
        raw.set_rectification(*cams)
        L, R, T, st = _c3_state(plain, cams, 9)
        k = len(T) - 1
        RL, RR = unrectify(L[k], cams[0]), unrectify(R[k], cams[1])
        args = (st, np.ones(len(st["uid"]), np.uint8), T[k], T[k - 1], T[k - 1], np.zeros(3), 1.2)
        want = fused(plain, rect(cams[0], RL), rect(cams[1], RR), *args)
        got = fused(raw, RL, RR, *args)
        assert_same(got, want, "rectified")
        assert want["source"] == "posit"


# ----------------------------------------------------------------------------------------------------------- C++ tracker
def _run_sv(tmp_path, L, R, mode):
    n = len(L)
    Lp, Rp = tmp_path / "L.raw", tmp_path / "R.raw"
    L.tofile(Lp)
    R.tofile(Rp)
    out = tmp_path / f"sv_{mode}.txt"
    env = dict(os.environ)
    env.pop("SVI_HOST_POSIT", None)
    if mode == "cpu":
        env["SVI_HOST_POSIT"] = "cpu"
    r = subprocess.run([str(EXE), "--sequence-sv", str(CALIB / "vi_sensor_left.txt"), str(CALIB / "vi_sensor_right.txt"), str(n), str(Lp), str(Rp),
                        "4000", str(out)], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    return out.read_text()


def _frames(text):
    return [dict(zip(w[2:-13:2], w[3:-13:2])) for w in (line.split() for line in text.splitlines()) if w[0] == "F"]


@pytest.mark.gpu
def test_cpp_tracker_fused_equals_composed_cpu_path(tmp_path):
    """facade_demo --sequence-sv prints the same bytes with the fused frame call (default) and with the composed calls and the CPU
    solve (SVI_HOST_POSIT=cpu): on a static camera, where the translation clamp keeps the pose at the detection pose and the
    regional search runs, and on the C3 sequence with three black frames, where the pose falls back to the prior and the solve
    takes over again afterwards."""
    from svi_mapper_b200.sequence import _render, make_world, render_sequence
    cams = _cams()
    W, H = cams[0].width, cams[0].height
    P_l, P_r = np.asarray(cams[0].P, np.float64).reshape(3, 4), np.asarray(cams[1].P, np.float64).reshape(3, 4)
    planes = make_world(cams[0], 4000)
    rng = np.random.default_rng(5)
    SL = np.stack([_render(planes, P_l, 0.0, np.eye(4), W, H, rng) for _ in range(12)])
    SR = np.stack([_render(planes, P_r, -P_r[0, 3] / P_r[0, 0], np.eye(4), W, H, rng) for _ in range(12)])
    fused_text = _run_sv(tmp_path, SL, SR, "gpu")
    assert fused_text == _run_sv(tmp_path, SL, SR, "cpu")
    assert any(int(f["S22"]) > 0 for f in _frames(fused_text)), fused_text[:2000]

    L, R, _ = render_sequence(cams[0], cams[1], 24, 4000)
    L[12:15] = 0
    R[12:15] = 0
    fused_text = _run_sv(tmp_path, L, R, "gpu")
    assert fused_text == _run_sv(tmp_path, L, R, "cpu")
    sources = [f["POSE"] for f in _frames(fused_text)]
    assert "prior" in sources[12:15] and "posit" in sources[15:], sources


@pytest.mark.gpu
def test_bounds_checked_build_sv_frame(tmp_path):
    """The parity tests of this file once against the -DSVI_BOUNDS_CHECK build: every new run-time index of the compaction,
    gather, assembly, routing and scatter kernels is asserted there, and a failed assertion fails the call.  The Python binding
    loads that build through SVI_GPU_LIB; facade_demo finds it as libsvi_gpu.so on LD_LIBRARY_PATH, which comes before its
    RUNPATH, so the fused C++ tracker runs its sequences against it too."""
    import shutil
    from svi_mapper_b200 import build as bld
    lib = bld.build_checked()
    libdir = tmp_path / "checked"
    libdir.mkdir()
    shutil.copy(lib, libdir / "libsvi_gpu.so")
    env = dict(os.environ, SVI_GPU_LIB=str(lib), LD_LIBRARY_PATH=os.pathsep.join(filter(None, [str(libdir), os.environ.get("LD_LIBRARY_PATH")])))
    r = subprocess.run([sys.executable, "-m", "pytest", str(pathlib.Path(__file__)), "-x", "-q", "-m", "gpu", "-k",
                        "composed_calls or rectification or cpp_tracker"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "3 passed" in r.stdout and "failed" not in r.stdout
