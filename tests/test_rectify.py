"""Undistortion + rectification of raw camera images (svi_rectify_map, svi_set_rectification, svi_rectify,
svi_multi_set_rectification; reference CStereoCamera.h:102-107: cv::initUndistortRectifyMap + cv::remap INTER_LINEAR).

CPU tier: the library's map and the numpy restatement (oracle/rectify_np.py) against cv2 byte for byte, the restated
fixed-point remap against cv2.remap, argument checks.  GPU tier: svi_rectify against cv2.remap, and every image entry point
on RAW images with rectification set against the same entry point on cv2-rectified images without it -- array by array,
byte for byte -- up to a 60-frame raw C3 sequence through the Python and the C++ tracker."""
import ctypes as C
import os
import pathlib
import subprocess
import sys

import numpy as np
import pytest

from oracle import rectify_np as rn
from svi_mapper_b200 import _lib
from svi_mapper_b200.calib import load_camera

ROOT = pathlib.Path(__file__).resolve().parents[1]
CALIB = ROOT / "tests" / "golden" / "calib"
RECTIFIABLE = [(n, s) for n in ("vi_sensor", "kitti_11_12") for s in ("left", "right")]


@pytest.fixture(scope="module")
def cv2_scalar():
    """cv2 with its scalar code paths on one thread, as the reference's maps were pinned."""
    import cv2
    opt, threads = cv2.useOptimized(), cv2.getNumThreads()
    cv2.setUseOptimized(False)
    cv2.setNumThreads(1)
    yield cv2
    cv2.setUseOptimized(opt)
    cv2.setNumThreads(threads)


def _cam(name, side):
    return load_camera(str(CALIB / f"{name}_{side}.txt"))


def _cv2_maps(cv2, cam, float_maps):
    args = (cam.K, cam.distortion, cam.rectification, cam.P, (cam.width, cam.height))
    if float_maps:
        return cv2.convertMaps(*cv2.initUndistortRectifyMap(*args, cv2.CV_32FC1), cv2.CV_16SC2)
    return cv2.initUndistortRectifyMap(*args, cv2.CV_16SC2)


# ----------------------------------------------------------------------------------------------------------- CPU tier
@pytest.mark.parametrize("float_maps", [False, True])
@pytest.mark.parametrize("name,side", RECTIFIABLE)
def test_library_map_equals_cv2(built_library, cv2_scalar, name, side, float_maps):
    from svi_mapper_b200.frontend import rectify_map
    cam = _cam(name, side)
    m1, m2 = _cv2_maps(cv2_scalar, cam, float_maps)
    xy, frac = rectify_map(cam, float_maps)
    assert xy.tobytes() == m1.tobytes() and frac.tobytes() == m2.tobytes()


@pytest.mark.parametrize("float_maps", [False, True])
@pytest.mark.parametrize("name,side", RECTIFIABLE)
def test_oracle_map_equals_cv2(cv2_scalar, name, side, float_maps):
    cam = _cam(name, side)
    m1, m2 = _cv2_maps(cv2_scalar, cam, float_maps)
    o1, o2 = rn.init_undistort_rectify_map(cam.K, cam.distortion, cam.rectification, cam.P, (cam.width, cam.height), float_maps)
    assert o1.tobytes() == m1.tobytes() and o2.tobytes() == m2.tobytes()


def test_map_saturates_far_coordinates_like_cv2(built_library, cv2_scalar):
    """A strongly distorted camera whose map leaves the int16 range: the integer parts saturate exactly as cv2 stores them
    (both map types).  The 5-bit fractions of this camera are not pinned: at sources 10^4 .. 10^7 px away the column step
    of cv2's loop (accumulated vs multiplied) shows in the last bit of u * 32; the calibrations of this repository agree to
    the last bit (test_library_map_equals_cv2)."""
    from svi_mapper_b200.calib import PinholeCamera
    from svi_mapper_b200.frontend import rectify_map
    cam = PinholeCamera("extreme", 96, 64, np.array([[20.0, 0, 48, 0], [0, 20, 32, 0], [0, 0, 1, 0]]),
                        np.array([[5e4, 0, 48], [0, 5e4, 32], [0, 0, 1.0]]), 0.0, np.array([3.0, 5.0, 0.1, -0.1]), np.eye(3))
    for float_maps in (False, True):
        m1, m2 = _cv2_maps(cv2_scalar, cam, float_maps)
        assert (m1 == 32767).any() and (m1 == -32768).any()
        xy, frac = rectify_map(cam, float_maps)
        assert xy.tobytes() == m1.tobytes()


def test_kitti_11_12_is_vi_sensor_optics_at_another_size():
    """kitti_11_12 ships the vi_sensor intrinsics, distortion and rectification at 1226 x 370: here it is a second image
    size for the map and the kernel, not a physically meaningful camera."""
    for side in ("left", "right"):
        a, b = _cam("kitti_11_12", side), _cam("vi_sensor", side)
        assert (a.width, a.height) == (1226, 370) and (b.width, b.height) == (752, 480)
        assert np.array_equal(a.K, b.K) and np.array_equal(a.distortion, b.distortion) and np.array_equal(a.rectification, b.rectification)
        assert a.distortion[0] < -0.2 and not np.array_equal(a.rectification, np.eye(3))


@pytest.mark.parametrize("side", ["left", "right"])
def test_kitti_00_has_no_calibration_and_is_refused(built_library, side):
    from svi_mapper_b200.frontend import SviError, rectify_map
    cam = _cam("kitti_00", side)
    assert not cam.K.any() and not cam.rectification.any()
    with pytest.raises(SviError) as e:
        rectify_map(cam)
    assert e.value.code == _lib.SVI_ERR_INVALID
    with pytest.raises(ValueError):
        rn.init_undistort_rectify_map(cam.K, cam.distortion, cam.rectification, cam.P, (cam.width, cam.height))


def test_interpolation_table_needs_no_fix_up():
    """initInterTab2D: rint(float32(1-t) * float32(1-t) * 32768) over all 1024 fractions is exact and sums to 32768, so
    OpenCV's sum fix-up never fires and the kernel's integer weights (32-fy or fy) * (32-fx or fx) * 32 are the table."""
    one = np.float32(1)
    for fy in range(32):
        for fx in range(32):
            ty, tx = np.float32(fy) * (one / np.float32(32)), np.float32(fx) * (one / np.float32(32))
            raw = np.rint(np.array([(one - ty) * (one - tx), (one - ty) * tx, ty * (one - tx), ty * tx], np.float32).astype(np.float64) * 32768)
            assert raw.sum() == 32768
            assert raw.tolist() == [(32 - fy) * (32 - fx) * 32, (32 - fy) * fx * 32, fy * (32 - fx) * 32, fy * fx * 32]
    assert np.array_equal(rn.inter_tab_2d().sum(-1), np.full((32, 32), 32768))


def test_oracle_remap_equals_cv2(cv2_scalar):
    """The restated fixed-point bilinear remap against cv2.remap: every one of the 1024 fractional positions, random images,
    and maps whose taps leave the image on every side (a tap outside reads 0, the others still count); then the vi_sensor
    and kitti_11_12 maps."""
    cv2 = cv2_scalar
    rng = np.random.default_rng(5)
    H, W = 64, 80
    for _ in range(3):
        img = rng.integers(0, 256, (H, W), dtype=np.uint8)
        frac = np.arange(H * W, dtype=np.int64).reshape(H, W) % 1024            # all 1024 fractions, 5 times over
        m2 = frac.astype(np.uint16)
        m1 = np.stack([rng.integers(-3, W + 2, (H, W)), rng.integers(-3, H + 2, (H, W))], -1).astype(np.int16)
        m1[0, :, 0], m1[1, :, 0], m1[2, :, 1], m1[3, :, 1] = -1, W - 1, -1, H - 1   # taps straddling each border
        m1[4, :4] = [[-32768, 0], [32767, 0], [0, -32768], [0, 32767]]
        assert rn.remap_linear(img, m1, m2).tobytes() == cv2.remap(img, m1, m2, cv2.INTER_LINEAR).tobytes()
        sat = img.copy()
        sat[:] = 255
        assert rn.remap_linear(sat, m1, m2).tobytes() == cv2.remap(sat, m1, m2, cv2.INTER_LINEAR).tobytes()
    for name, side in RECTIFIABLE:
        cam = _cam(name, side)
        m1, m2 = _cv2_maps(cv2, cam, False)
        img = rng.integers(0, 256, (cam.height, cam.width), dtype=np.uint8)
        assert rn.remap_linear(img, m1, m2).tobytes() == cv2.remap(img, m1, m2, cv2.INTER_LINEAR).tobytes()


def test_new_entry_points_refuse_a_null_context(built_library):
    lib = _lib.load()
    r = _lib.Rectification()
    img = np.zeros((64, 64), np.uint8)
    assert lib.svi_set_rectification(None, C.byref(r), C.byref(r)) == _lib.SVI_ERR_INVALID
    assert lib.svi_set_rectification(None, None, None) == _lib.SVI_ERR_INVALID
    assert lib.svi_rectify(None, 0, img.ctypes.data, 64, 64 * 64, 1, img.ctypes.data, 64) == _lib.SVI_ERR_INVALID
    assert lib.svi_multi_set_rectification(None, C.byref(r), C.byref(r)) == _lib.SVI_ERR_INVALID
    assert lib.svi_rectify_map(None, C.byref(r), img.ctypes.data, img.ctypes.data) == _lib.SVI_ERR_INVALID


# ----------------------------------------------------------------------------------------------------------- GPU tier
def _raw_pair(cams, seed):
    """A raw (distorted, unrectified) stereo pair: the synthetic rectified pair seen through the calibrated optics."""
    from svi_mapper_b200.synth import stereo_pair, unrectify
    L, R = stereo_pair(cams[0].width, cams[0].height, seed)
    return unrectify(L, cams[0]), unrectify(R, cams[1])


def _cv2_rectify(cv2, cam, raw, float_maps=False):
    m1, m2 = _cv2_maps(cv2, cam, float_maps)
    if raw.ndim == 2:
        return cv2.remap(raw, m1, m2, cv2.INTER_LINEAR)
    return np.stack([cv2.remap(r, m1, m2, cv2.INTER_LINEAR) for r in raw])


def _same_frames(a, b, n):
    assert a.n_keypoints.tobytes() == b.n_keypoints.tobytes() and a.n_detected.tobytes() == b.n_detected.tobytes()
    assert a.n_keypoints.min() > 100
    for f in range(n):
        _same_new(a.frame(f), b.frame(f))


def _same_new(x, y):
    """New-landmark results as svi_stereo_result specifies them: every array over the live key-points, the RIGHT-side
    match (uv_r, desc_r, xyz) where the status is SVI_OK -- the library leaves those slots unspecified otherwise."""
    assert x.keys() == y.keys()
    for k in ("uv_l", "desc_l", "status", "dist", "idx"):
        assert x[k].shape == y[k].shape and x[k].tobytes() == y[k].tobytes(), k
    ok = x["status"] == 0
    assert ok.sum() > 10
    for k in ("uv_r", "desc_r", "xyz"):
        assert x[k][ok].tobytes() == y[k][ok].tobytes(), k


def _same_dict(x, y):
    """Per-query results (triangulation, tracking): the library writes every slot, so every byte is compared."""
    assert x.keys() == y.keys()
    for k in x:
        assert x[k].shape == y[k].shape and x[k].tobytes() == y[k].tobytes(), k


@pytest.mark.gpu
@pytest.mark.parametrize("float_maps", [False, True])
@pytest.mark.parametrize("cams_name", ["vi_cams", "kitti1112_cams"])
def test_svi_rectify_equals_cv2_remap(request, built_library, cv2_scalar, cams_name, float_maps):
    from svi_mapper_b200 import StereoFrontend
    cams = request.getfixturevalue(cams_name)
    W, H = cams[0].width, cams[0].height
    rng = np.random.default_rng(9)
    raw = rng.integers(0, 256, (7, H, W), dtype=np.uint8)
    raw[1] = _raw_pair(cams, 4000)[0]
    with StereoFrontend(*cams, chunk_frames=3) as fe:
        fe.set_rectification(*cams, float_maps=float_maps)
        for side in (0, 1):
            want = _cv2_rectify(cv2_scalar, cams[side], raw, float_maps)
            for n in (1, 2, 7):                                                  # 7: three chunks of 3
                assert fe.rectify(raw[:n], side).tobytes() == want[:n].tobytes(), (side, n)
            assert fe.rectify(raw[3], side).tobytes() == want[3].tobytes()
            # pitch > W on both sides of the call, frames not densely stacked on the way in
            pitch, opitch = W + 37, W + 5
            src = np.zeros((4, H + 2, pitch), np.uint8)
            src[:, :H, :W] = raw[:4]
            out = np.full((4, H, opitch), 7, np.uint8)
            rc = fe._lib.svi_rectify(fe._ctx, side, src.ctypes.data, pitch, (H + 2) * pitch, 4, out.ctypes.data, opitch)
            assert rc == 0
            assert out[:, :, :W].tobytes() == want[:4].tobytes() and (out[:, :, W:] == 7).all()


@pytest.mark.gpu
def test_new_landmark_entry_points_on_raw_images(built_library, cv2_scalar, vi_cams):
    """svi_stereo_frames (small-call and batch path, with masks), svi_stereo_frames_device (dense and padded rows),
    svi_stereo_frame_masked: raw images + rectification == cv2-rectified images without it, byte for byte."""
    import torch
    from svi_mapper_b200 import StereoFrontend
    W, H = vi_cams[0].width, vi_cams[0].height
    pairs = [_raw_pair(vi_cams, 4000 + i) for i in range(6)]
    RL, RR = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    L, R = _cv2_rectify(cv2_scalar, vi_cams[0], RL), _cv2_rectify(cv2_scalar, vi_cams[1], RR)
    masks = np.full((6, H, W), 255, np.uint8)
    masks[::2, 100:220, 200:500] = 0
    with StereoFrontend(*vi_cams, chunk_frames=4) as plain, StereoFrontend(*vi_cams, chunk_frames=4) as fe:
        k0 = fe.kernels_per_chunk(6), fe.kernels_per_chunk(1)
        fe.set_rectification(*vi_cams)
        assert (fe.kernels_per_chunk(6), fe.kernels_per_chunk(1)) == (k0[0] + 1, k0[1] + 1)
        for n in (1, 2, 6):                                                     # 1, 2: small-call path; 6: two batch chunks
            _same_frames(fe.stereo_frames(RL[:n], RR[:n]), plain.stereo_frames(L[:n], R[:n]), n)
            _same_frames(fe.stereo_frames(RL[:n], RR[:n], masks[:n]), plain.stereo_frames(L[:n], R[:n], masks[:n]), n)
        centres = np.array([[100.5, 80.2], [400.0, 300.0], [600.7, 50.1]], np.float32)
        _same_new(fe.add_new_landmarks(RL[0], RR[0], mask_centres=centres), plain.add_new_landmarks(L[0], R[0], mask_centres=centres))
        _same_new(fe.add_new_landmarks(RL[1], RR[1], mask_centres=np.zeros((0, 2))), plain.add_new_landmarks(L[1], R[1], mask_centres=np.zeros((0, 2))))

        def device_run(front, a, b, m, pad):
            n, cap = a.shape[0], front.max_corners
            pitch = W + pad

            def up(x):
                t = torch.zeros((n, H, pitch), dtype=torch.uint8, device="cuda")
                t[:, :, :W] = torch.from_numpy(x)
                return t
            ta, tb, tm = up(a), up(b), up(m)
            o = dict(n_keypoints=torch.zeros(n, dtype=torch.int32), n_detected=torch.zeros(n, dtype=torch.int32),
                     uv_left=torch.zeros((n, cap, 2)), uv_right=torch.zeros((n, cap, 2)), xyz_left=torch.zeros((n, cap, 3), dtype=torch.float64),
                     desc_left=torch.zeros((n, cap, 32), dtype=torch.uint8), desc_right=torch.zeros((n, cap, 32), dtype=torch.uint8),
                     distance=torch.zeros((n, cap), dtype=torch.int32), match_index=torch.zeros((n, cap), dtype=torch.int32),
                     status=torch.zeros((n, cap), dtype=torch.uint8))
            o = {k: v.cuda() for k, v in o.items()}
            r = _lib.StereoResult(cap, *(o[k].data_ptr() for k in ("n_keypoints", "n_detected", "uv_left", "uv_right", "xyz_left", "desc_left",
                                                                   "desc_right", "distance", "match_index", "status")))
            front.stereo_frames_device(ta.data_ptr(), tb.data_ptr(), pitch, H * pitch, n, r, tm.data_ptr())
            torch.cuda.synchronize()
            front.check_overflow()
            from svi_mapper_b200 import StereoFrames
            return StereoFrames(**{k: v.cpu().numpy() for k, v in o.items()})

        for pad in (0, 40):
            _same_frames(device_run(fe, RL, RR, masks, pad), device_run(plain, L, R, masks, pad), 6)


def _track_state(plain, L, R):
    d = plain.add_new_landmarks(L, R)
    ok = np.nonzero(d["status"] == 0)[0][:300]
    assert len(ok) > 100
    disp = (d["uv_l"][ok, 0] - d["uv_r"][ok, 0]).astype(np.float32)
    return d, ok, disp


@pytest.mark.gpu
def test_query_entry_points_on_raw_images(built_library, cv2_scalar, vi_cams):
    """svi_harris_response, svi_detect, svi_describe (LEFT), svi_triangulate_right / _left and svi_track_landmarks with all
    three stages and each _stages subset: raw images + rectification == cv2-rectified images without it."""
    from svi_mapper_b200 import StereoFrontend
    from svi_mapper_b200.synth import stereo_pair, unrectify
    W, H = vi_cams[0].width, vi_cams[0].height
    L0, R0 = stereo_pair(W, H, 4000)
    L1, R1 = np.roll(L0, (2, 3), axis=(0, 1)), np.roll(R0, (2, 3), axis=(0, 1))
    raw = [unrectify(x, vi_cams[i % 2]) for i, x in enumerate((L0, R0, L1, R1))]
    rect = [_cv2_rectify(cv2_scalar, vi_cams[i % 2], x) for i, x in enumerate(raw)]
    with StereoFrontend(*vi_cams) as plain, StereoFrontend(*vi_cams) as fe:
        fe.set_rectification(*vi_cams)
        assert fe.harris_response(raw[0]).tobytes() == plain.harris_response(rect[0]).tobytes()
        mask = np.full((H, W), 255, np.uint8)
        mask[50:200, 100:300] = 0
        for a, b in zip(fe.detect(np.stack([raw[0], raw[2]]), np.stack([mask, mask])), plain.detect(np.stack([rect[0], rect[2]]), np.stack([mask, mask]))):
            assert a.tobytes() == b.tobytes() and len(a) > 100
        d, ok, disp = _track_state(plain, rect[0], rect[1])
        for x, y in zip(fe.describe(raw[2], d["uv_l"][ok]), plain.describe(rect[2], d["uv_l"][ok])):
            assert x.tobytes() == y.tobytes()
        tl = np.stack([np.maximum(np.float32(0), d["uv_l"][ok, 0] - np.float32(28 + 60)), d["uv_l"][ok, 1] - np.float32(28)], 1)
        tr_f = fe.triangulate_right(raw[3], tl, d["uv_l"][ok], d["desc_l"][ok])
        tr_p = plain.triangulate_right(rect[3], tl, d["uv_l"][ok], d["desc_l"][ok])
        _same_dict(tr_f, tr_p)
        assert (tr_p["status"] == 0).sum() > 50
        sr = np.full(len(ok), 60.0, np.float32)
        tl = (d["uv_r"][ok] - np.float32(28)).astype(np.float32)
        tl_f = fe.triangulate_left(raw[2], sr, tl, d["uv_r"][ok], d["desc_r"][ok])
        _same_dict(tl_f, plain.triangulate_left(rect[2], sr, tl, d["uv_r"][ok], d["desc_r"][ok]))
        assert (tl_f["status"] == 0).sum() > 50
        T = np.eye(4)
        T[:3, 3] = (0.015, 0.01, 0.0)
        seen = np.zeros(6, int)
        for (a, b), pose, scaling, stages in (((0, 1), T, 1.0, None), ((2, 3), np.eye(4), 1.0, None), ((0, 1), T, 1.0, 1), ((2, 3), np.eye(4), 1.0, 2),
                                             ((2, 3), np.eye(4), 1.0, 3), ((0, 1), T, 1.5, 4), ((2, 3), T, 1.5, 7), ((2, 3), T, 1.5, 6)):
            args = (pose, d["xyz"][ok], d["desc_l"][ok], d["desc_r"][ok], disp, 7.0, scaling)
            kw = dict(uv_reference_left=d["uv_l"][ok], desc_reference_left=d["desc_l"][ok], T_left_to_world_at_detection=np.eye(4), stages=stages)
            got, want = fe.track_landmarks(raw[a], raw[b], *args, **kw), plain.track_landmarks(rect[a], rect[b], *args, **kw)
            _same_dict(got, want)
            seen += np.bincount(want["stage"], minlength=6)
        assert seen[1] > 20 and seen[3] + seen[4] > 20 and seen[5] > 20, seen


@pytest.mark.gpu
def test_clearing_rectification_restores_the_plain_context(built_library, cv2_scalar, vi_cams):
    from svi_mapper_b200 import StereoFrontend
    from svi_mapper_b200.frontend import SviError
    RL, RR = _raw_pair(vi_cams, 4100)
    L, R = _cv2_rectify(cv2_scalar, vi_cams[0], RL), _cv2_rectify(cv2_scalar, vi_cams[1], RR)
    with StereoFrontend(*vi_cams) as never:
        want = never.stereo_frames(np.stack([L, L]), np.stack([R, R]))
        want_one = never.add_new_landmarks(L, R, mask_centres=np.array([[300.0, 200.0]]))
        k = never.kernels_per_chunk(64)
    with StereoFrontend(*vi_cams) as fe:
        for float_maps in (True, False):
            fe.set_rectification(*vi_cams, float_maps=float_maps)
        _same_frames(fe.stereo_frames(np.stack([RL, RL]), np.stack([RR, RR])), want, 2)
        fe.clear_rectification()
        fe.clear_rectification()
        assert fe.kernels_per_chunk(64) == k
        _same_frames(fe.stereo_frames(np.stack([L, L]), np.stack([R, R])), want, 2)
        _same_new(fe.add_new_landmarks(L, R, mask_centres=np.array([[300.0, 200.0]])), want_one)
        with pytest.raises(SviError):
            fe.rectify(RL, 0)                                                     # nothing set
        kitti = (_cam("kitti_00", "left"), _cam("kitti_00", "right"))
        with pytest.raises(SviError) as e:
            fe.set_rectification(*kitti)
        assert e.value.code == _lib.SVI_ERR_INVALID
        _same_frames(fe.stereo_frames(np.stack([L, L]), np.stack([R, R])), want, 2)   # a refused calibration changes nothing


@pytest.mark.gpu
def test_multi_driver_with_rectification_equals_one_context(built_library, vi_cams):
    from svi_mapper_b200 import MultiFrontend, StereoFrontend
    pairs = [_raw_pair(vi_cams, 4200 + i) for i in range(3)]
    n = 11
    RL, RR = np.stack([pairs[i % 3][0] for i in range(n)]), np.stack([pairs[i % 3][1] for i in range(n)])
    for i in range(n):
        RL[i, :, : 8 + i] = RL[i, :, : 8 + i][:, ::-1]
    with StereoFrontend(*vi_cams, chunk_frames=4) as fe:
        fe.set_rectification(*vi_cams)
        one = fe.stereo_frames(RL, RR)
    with MultiFrontend(*vi_cams, devices=[0, 0], chunk_frames=4) as mf:
        mf.set_rectification(*vi_cams)
        _same_frames(mf.stereo_frames(RL, RR), one, n)


def _raw_sequence(cams, n, seed):
    from svi_mapper_b200.sequence import render_sequence
    from svi_mapper_b200.synth import unrectify
    L, R, T = render_sequence(cams[0], cams[1], n, seed)
    return np.stack([unrectify(x, cams[0]) for x in L]), np.stack([unrectify(x, cams[1]) for x in R]), T


@pytest.mark.gpu
def test_raw_c3_sequence_tracks_as_the_cv2_rectified_one(built_library, cv2_scalar, vi_cams):
    """BASELINE configs[2] on raw frames: the 60-frame vi_sensor sequence rendered through the distorted optics, run through
    SequenceTracker + GpuBackend with rectification on, against the cv2-rectified frames without it: every frame's log
    record, tracking result, new-landmark result and the landmark state are identical."""
    from svi_mapper_b200 import StereoFrontend
    from svi_mapper_b200.sequence import GpuBackend, SequenceTracker
    n = 60
    RL, RR, T = _raw_sequence(vi_cams, n, 4000)
    L, R = _cv2_rectify(cv2_scalar, vi_cams[0], RL), _cv2_rectify(cv2_scalar, vi_cams[1], RR)
    with StereoFrontend(*vi_cams) as fe, StereoFrontend(*vi_cams) as plain:
        fe.set_rectification(*vi_cams)
        a, b = SequenceTracker(GpuBackend(fe), vi_cams[0]), SequenceTracker(GpuBackend(plain), vi_cams[0])
        for t in range(n):
            ra, rb = a.process(RL[t], RR[t], T[t]), b.process(L[t], R[t], T[t])
            assert ra == rb, (t, ra, rb)
            if ra["tracked"]:
                _same_dict(a.last_track, b.last_track)
            for k in a.s:
                assert a.s[k].tobytes() == b.s[k].tobytes(), (t, k)
    stages = np.sum([r["stages"] for r in a.log], axis=0)
    assert a.n_active > 500 and stages[1] > 1000 and stages[5] > 50 and sum(r["new"] > 0 for r in a.log) >= 3, (a.n_active, stages)


@pytest.mark.gpu
def test_cpp_tracker_on_raw_frames(built_library, cv2_scalar, vi_cams, tmp_path):
    """facade_demo --sequence with --rectify (CGpuContext::setRectification from the CPinholeCamera members) on raw frames
    prints exactly what it prints for the cv2-rectified frames without it."""
    n, mc = 12, 150
    RL, RR, T = _raw_sequence(vi_cams, n, 4100)
    L, R = _cv2_rectify(cv2_scalar, vi_cams[0], RL), _cv2_rectify(cv2_scalar, vi_cams[1], RR)
    with open(tmp_path / "motions.txt", "w") as f:
        for t in range(n):
            M = np.eye(4) if t == 0 else T[t] @ np.linalg.inv(T[t - 1])
            f.write(" ".join(repr(float(v)) for v in M[:3].reshape(-1)) + " " + repr(float(np.arccos(np.clip((np.trace(M[:3, :3]) - 1.0) / 2.0, -1.0, 1.0)))) + "\n")
    exe = ROOT / "svi_mapper_b200" / "host" / "facade_demo"
    outs = []
    for tag, a, b, flag in (("raw", RL, RR, ["--rectify"]), ("rect", L, R, [])):
        a.tofile(tmp_path / f"L_{tag}.raw")
        b.tofile(tmp_path / f"R_{tag}.raw")
        out = tmp_path / f"seq_{tag}.txt"
        r = subprocess.run([str(exe), "--sequence", *flag, str(CALIB / "vi_sensor_left.txt"), str(CALIB / "vi_sensor_right.txt"), str(n),
                            str(tmp_path / f"L_{tag}.raw"), str(tmp_path / f"R_{tag}.raw"), str(tmp_path / "motions.txt"), str(mc), str(out)],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        outs.append(out.read_text())
    assert outs[0] == outs[1] and outs[0].count("\nA ") > 200


@pytest.mark.gpu
def test_bounds_checked_build_on_raw_images(built_library):
    """The GPU tests of this file once against the -DSVI_BOUNDS_CHECK build: every map, tap and output index of
    rectify_kernel is asserted there, and so are the pipeline kernels that read the rectified planes."""
    from svi_mapper_b200 import build as bld
    lib = bld.build_checked()
    k = "not bounds_checked and not c3_sequence and not cpp_tracker"
    r = subprocess.run([sys.executable, "-m", "pytest", str(pathlib.Path(__file__)), "-x", "-q", "-m", "gpu", "-k", k], env=dict(os.environ, SVI_GPU_LIB=str(lib)),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "failed" not in r.stdout
