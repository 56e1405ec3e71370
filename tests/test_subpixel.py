"""Sub-pixel disparity (svi_params.subpixel_window / subpixel_search): SAD patch refinement of every SVI_OK match, on the device.

CPU tier: the CPU restatement of the refinement (tests/subpixel_np.py) recovers a known fractional shift, lowers the depth
error of the rendered vi_sensor sequence against the renderer's exact depth, and follows the status rules on hand-built
patches.  GPU tier: every entry point with the mode on equals the restatement's refinement of the same call with the mode off, bit
for bit (status, uv_right, xyz_left), and leaves every other field byte-identical; the mode off equals the default ctx;
invalid (w, L) are refused; the launch count, the stage timings, and a rerun against the bounds-checked build."""
import os
import pathlib
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import frontend_np as o
import subpixel_np as sp
from svi_mapper_b200.synth import left_image, stereo_pair

F32 = np.float32
ROOT = pathlib.Path(__file__).resolve().parents[1]
WL = [(1, 1), (5, 5), (12, 16)]


def _tri(cams, **kw):
    cl, cr = cams
    return o.Triangulator(o.Camera(cl.width, cl.height, np.asarray(cl.P, np.float64).reshape(3, 4)),
                          o.Camera(cr.width, cr.height, np.asarray(cr.P, np.float64).reshape(3, 4)), o.StereoParams(**kw))


def _sized(cams, W, H):
    return tuple(SimpleNamespace(width=W, height=H, P=c.P) for c in cams)


# ------------------------------------------------------------------------------------------------------------ CPU tier
def test_restatement_recovers_a_fractional_shift(vi_cams):
    """RIGHT = LEFT resampled 17.3 px to the left (linear interpolation): from the integer match at 17 px the refined
    disparity is within 0.15 px of 17.3 for most slots (the parabola through SAD values is biased towards whole pixels,
    so not for all), and the depth follows from it."""
    W, H, d = 400, 240, 17.3
    big = left_image(W + 40, H, 5).astype(np.float64)
    x = np.arange(W) + d
    x0 = np.floor(x).astype(int)
    a = x - x0
    R = np.clip(np.rint(big[:, x0] * (1 - a) + big[:, x0 + 1] * a), 0, 255).astype(np.uint8)
    L = big[:, :W].astype(np.uint8)
    tri = _tri(_sized(vi_cams, W, H))
    ys, xs = np.meshgrid(np.arange(40, H - 40, 9), np.arange(60, W - 40, 9), indexing="ij")
    uv_l = np.stack([xs.ravel(), ys.ravel()], 1).astype(F32)
    uv_r = uv_l - F32([17, 0])
    st = np.zeros(len(uv_l), np.uint8)
    ur, xyz, st2 = sp.subpixel_refine(L, R, uv_l, uv_r, st, 5, 5, tri)
    ok = st2 == o.ST_OK
    assert ok.mean() > 0.95
    err = np.abs((uv_l[ok, 0] - ur[ok, 0]) - d)
    assert (err < 0.15).mean() > 0.6 and err.max() < 0.5, np.quantile(err, [0.5, 0.8, 1.0])
    np.testing.assert_array_equal(ur[:, 1], uv_r[:, 1])
    np.testing.assert_allclose(xyz[ok, 2], tri.du_r_flipped / (uv_l[ok, 0] - ur[ok, 0]).astype(np.float64), rtol=1e-12)


def _true_depth(planes, cam, T, uv):
    """Depth of the renderer's nearest visible plane along the LEFT ray through each pixel (svi_mapper_b200.sequence._render)."""
    P = np.asarray(cam.P, np.float64).reshape(3, 4)
    f, cx, cy = P[0, 0], P[0, 2], P[1, 2]
    R, t = T[:3, :3], T[:3, 3]
    ray_w = np.stack([(uv[:, 0] - cx) / f, (uv[:, 1] - cy) / f, np.ones(len(uv))], -1) @ R
    c_w = (-t) @ R
    z = np.full(len(uv), np.nan)
    for pl in planes:   # far -> near, as the renderer paints them
        s = (pl["z"] - c_w[2]) / ray_w[:, 2]
        tx = (c_w[0] + s * ray_w[:, 0] - pl["x0"]) / pl["texel"]
        ty = (c_w[1] + s * ray_w[:, 1] - pl["y0"]) / pl["texel"]
        th, tw = pl["tex"].shape
        hit = (s > 0) & (tx >= 0) & (ty >= 0) & (tx < tw - 1) & (ty < th - 1)
        z = np.where(hit, s, z)   # camera-frame depth: the ray has z = 1 in the camera frame
    return z


def test_restatement_lowers_depth_error_on_the_rendered_sequence(vi_cams):
    """Frames 0 and 30 of the rendered vi_sensor sequence: median relative depth error against the renderer's depth at least
    2x lower with refinement (w = L = 5) for 0-5 m and 5-15 m, and not higher for 15-30 m and 30-50 m."""
    from svi_mapper_b200.sequence import make_world, render_sequence
    cl, cr = vi_cams
    L, R, T = render_sequence(cl, cr, 31, 4000)
    planes = make_world(cl, 4000)
    tri = _tri(vi_cams)
    for fr in (0, 30):
        base = o.add_new_landmarks(L[fr], R[fr], tri)
        sub = sp.add_new_landmarks(L[fr], R[fr], tri, subpixel=(5, 5))
        for k in ("uv_l", "desc_l", "dist", "idx"):
            np.testing.assert_array_equal(sub[k], base[k])
        ok = (base["status"] == o.ST_OK) & (sub["status"] == o.ST_OK)
        rejected = (base["status"] == o.ST_OK) & (sub["status"] == sp.ST_SUBPIXEL_REJECTED)
        assert ok.sum() > 700 and rejected.sum() < 0.03 * (base["status"] == o.ST_OK).sum()
        z = _true_depth(planes, cl, T[fr], base["uv_l"][ok].astype(np.float64))
        e_int = np.abs(base["xyz"][ok, 2] - z) / z
        e_sub = np.abs(sub["xyz"][ok, 2] - z) / z
        for lo, hi, factor in ((0, 5, 2.0), (5, 15, 2.0), (15, 30, 1.0), (30, 50, 1.0)):
            m = (z >= lo) & (z < hi)
            assert m.sum() > 40, (fr, lo, hi)
            assert np.median(e_sub[m]) * factor <= np.median(e_int[m]), (fr, lo, hi, np.median(e_int[m]), np.median(e_sub[m]))


def test_restatement_status_rules_on_hand_built_patches(vi_cams):
    """k* = +-L is SVI_SUBPIXEL_REJECTED; a tie between two minima takes the first; w + L = 28 at the border-most position
    BRIEF's filter keeps reads only inside the image; a refined disparity of 0 is SVI_TRI_ZERO_DISP; slots that are not
    SVI_OK are left alone."""
    tri = _tri(_sized(vi_cams, 120, 80))
    rng = np.random.default_rng(3)
    img_l = rng.integers(0, 256, (80, 120), dtype=np.uint8)
    uv_l = np.array([[70, 40]], F32)
    for shift, want in ((0, o.ST_OK), (2, o.ST_OK), (-2, o.ST_OK), (3, sp.ST_SUBPIXEL_REJECTED), (-3, sp.ST_SUBPIXEL_REJECTED)):
        img_r = np.roll(img_l, -40 + shift, axis=1)          # LEFT (70, 40) is RIGHT (30 + shift, 40): SAD(shift) = 0
        ur, xyz, st = sp.subpixel_refine(img_l, img_r, uv_l, np.array([[30, 40]], F32), [0], 4, 3, tri)
        assert st[0] == want, shift
        if want == o.ST_OK:
            assert abs(float(ur[0, 0]) - (30 + shift)) < 0.5
            assert xyz[0, 2] == tri.du_r_flipped / float(F32(70) - ur[0, 0])
    # tie: columns of period 2 on both sides; RIGHT (31, 40) has the LEFT patch at k = -1 and k = +1, SAD(-2) == SAD(0)
    col = rng.integers(0, 256, (80, 2), dtype=np.uint8)
    per = np.tile(col, (1, 60))
    ur, _, st = sp.subpixel_refine(per, per, uv_l, np.array([[31, 40]], F32), [0], 3, 2, tri)
    assert st[0] == o.ST_OK and ur[0, 0] == F32(30)          # the first minimum (k* = -1) and delta = 0
    # w + L = 28 at 28 px from the left edge of RIGHT and the top edge: every index inside the image
    img_r = np.roll(img_l, -63, axis=1)                        # LEFT (91, 28) is RIGHT (28, 28)
    for w, Lr in ((27, 1), (1, 27), (14, 14)):
        ur, _, st = sp.subpixel_refine(img_l, img_r, np.array([[91, 28]], F32), np.array([[28, 28]], F32), [0], w, Lr, tri)
        assert st[0] == o.ST_OK and abs(float(ur[0, 0]) - 28) < 0.5, (w, Lr)
    # a patch mirror-symmetric about the match: SAD(-1) == SAD(+1), delta = 0, and zero disparity
    sym = rng.integers(0, 256, (80, 120), dtype=np.uint8)
    sym[:, 61:] = sym[:, 59:0:-1][:, :59]
    ur, _, st = sp.subpixel_refine(sym, sym, np.array([[60, 40]], F32), np.array([[60, 40]], F32), [0], 3, 2, tri)
    assert st[0] == o.ST_TRI_ZERO_DISP
    # other statuses pass through untouched
    ur, xyz, st = sp.subpixel_refine(img_l, img_l, np.array([[60, 40]] * 3, F32), np.array([[9, 9]] * 3, F32),
                                    [o.ST_TRI_DISTANCE, o.ST_TRI_ZERO_DISP, sp.ST_SPARSE_NOT_MUTUAL], 5, 5, tri)
    assert list(st) == [o.ST_TRI_DISTANCE, o.ST_TRI_ZERO_DISP, sp.ST_SPARSE_NOT_MUTUAL] and (ur == 9).all() and (xyz == 0).all()


# ------------------------------------------------------------------------------------------------------------ GPU tier
def _fe(cams, **kw):
    from svi_mapper_b200 import StereoFrontend
    return StereoFrontend(*cams, **kw)


UNCHANGED = ("uv_l", "desc_l", "dist", "idx")


def assert_refined(on: dict, off: dict, L, R, tri, w, Lr, what=""):
    """`on` (mode on) == the restatement's refinement of `off` (mode off, same call): status, uv_right and xyz_left bit for bit;
    desc_right, uv_right.y and every other field as with the mode off."""
    assert len(on["uv_l"]) == len(off["uv_l"]), what
    for k in UNCHANGED + (("second",) if "second" in off else ()):
        np.testing.assert_array_equal(on[k], off[k], err_msg=f"{what} {k}")
    if "n_right" in off:
        assert on["n_right"] == off["n_right"]
    uv_r, xyz, st = sp.subpixel_refine(L, R, off["uv_l"], off["uv_r"], off["status"], w, Lr, tri)
    np.testing.assert_array_equal(on["status"], st, err_msg=f"{what} status")
    ok = st == o.ST_OK
    np.testing.assert_array_equal(on["uv_r"][ok], uv_r[ok], err_msg=f"{what} uv_r")
    np.testing.assert_array_equal(on["xyz"][ok], xyz[ok], err_msg=f"{what} xyz")
    np.testing.assert_array_equal(on["desc_r"][ok], off["desc_r"][ok], err_msg=f"{what} desc_r")
    return int(ok.sum()), int((st == sp.ST_SUBPIXEL_REJECTED).sum()), int((uv_r[ok, 0] != np.rint(uv_r[ok, 0])).sum())


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
@pytest.mark.parametrize("shape", ["c2_binned", "c4_per_keypoint"])
def test_dense_batch_equals_restatement(monkeypatch, kitti_cams, kitti1112_cams, shape):
    """26 frames in one chunk (the batch path): C2's shape with the binned matcher, C4's density with the per-key-point
    matcher; three (w, L); one more launch per chunk."""
    monkeypatch.setenv("SVI_MATCH_BINNED", "2" if shape == "c2_binned" else "1")
    cams, mc = (kitti_cams, 2000) if shape == "c2_binned" else (kitti1112_cams, 1000)
    W, H = cams[0].width, cams[0].height
    pairs = [stereo_pair(W, H, 7000 + i) for i in range(26)]
    Ls, Rs = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    tri = _tri(cams)
    with _fe(cams, max_corners=mc, chunk_frames=26) as off:
        k_off = off.kernels_per_chunk(26)
        assert k_off == (6 if shape == "c2_binned" else 5)
        base = off.stereo_frames(Ls, Rs)
    for w, Lr in WL:
        with _fe(cams, max_corners=mc, chunk_frames=26, subpixel_window=w, subpixel_search=Lr) as fe:
            assert fe.kernels_per_chunk(26) == k_off + 1
            res = fe.stereo_frames(Ls, Rs)
            np.testing.assert_array_equal(res.n_keypoints, base.n_keypoints)
            np.testing.assert_array_equal(res.n_detected, base.n_detected)
            for f in range(26):
                got, ref = res.frame(f), base.frame(f)
                for k in UNCHANGED:
                    np.testing.assert_array_equal(got[k], ref[k])
                if f in (0, 13, 25):
                    n_ok, n_rej, n_frac = assert_refined(got, ref, Ls[f], Rs[f], tri, w, Lr, f"{shape} {w},{Lr} frame {f}")
                    assert n_ok > 300 and n_frac > 0.5 * n_ok


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_c5_long_scan_line(kitti_cams):
    """One 3840 x 1080 pair, 10 k corners, 1000-px scan lines."""
    W, H = 3840, 1080
    cams = _sized(kitti_cams, W, H)
    L, R = stereo_pair(W, H, 3000, d_max=900)
    kw = dict(max_corners=10000, search_range_px=1000.0, max_candidates=131072, chunk_frames=1)
    with _fe(cams, **kw) as off, _fe(cams, subpixel_window=5, subpixel_search=5, **kw) as fe:
        n_ok, _, _ = assert_refined(fe.stereo_frames(L, R).frame(0), off.stereo_frames(L, R).frame(0), L, R, _tri(cams), 5, 5, "C5")
        assert n_ok > 5000


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_masked_frame_equals_full_restatement(vi_cams):
    """svi_stereo_frame_masked (the one-pair path, mask built from landmark centres) against the oracle's addNewLandmarks
    followed by the refinement, end to end, and against the mode-off call."""
    W, H = 376, 240
    cams = _sized(vi_cams, W, H)
    L, R = stereo_pair(W, H, 41)
    centres = np.random.default_rng(2).uniform([0, 0], [W, H], (60, 2)).astype(F32)
    tri = _tri(cams)
    ref = sp.add_new_landmarks(L, R, tri, mask=o.mask_active_landmarks(W, H, centres), subpixel=(5, 5))
    with _fe(cams) as off, _fe(cams, subpixel_window=5, subpixel_search=5) as fe:
        got = fe.add_new_landmarks(L, R, mask_centres=centres)
        base = off.add_new_landmarks(L, R, mask_centres=centres)
        assert_refined(got, base, L, R, tri, 5, 5, "masked")
        for k in UNCHANGED + ("status",):
            np.testing.assert_array_equal(got[k], ref[k], err_msg=k)
        ok = ref["status"] == o.ST_OK
        assert ok.sum() > 100
        for k in ("uv_r", "xyz", "desc_r"):
            np.testing.assert_array_equal(got[k][ok], ref[k][ok], err_msg=k)


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
@pytest.mark.parametrize("mutual", [0, 1])
def test_sparse_frames_equal_restatement(kitti_cams, mutual):
    """Sparse frames (five frames in chunks of two), two bands, with and without the left-right check; the refined result
    also equals the numpy restatement of a sparse frame with the refinement applied."""
    from test_sparse_frames import sparse_frame_np
    W, H = kitti_cams[0].width, kitti_cams[0].height
    pairs = [stereo_pair(W, H, 510 + i) for i in range(5)]
    Ls, Rs = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    tri = _tri(kitti_cams)
    with _fe(kitti_cams, chunk_frames=2) as off, _fe(kitti_cams, chunk_frames=2, subpixel_window=5, subpixel_search=5) as fe:
        for band in ((1.0, 1.0, 60.0), (1e9, -1e9, 1e9)):
            res = fe.stereo_frames_sparse(Ls, Rs, None, *band, mutual=bool(mutual))
            base = off.stereo_frames_sparse(Ls, Rs, None, *band, mutual=bool(mutual))
            np.testing.assert_array_equal(res.n_keypoints_right, base.n_keypoints_right)
            for f in range(5):
                assert_refined(res.frame(f), base.frame(f), Ls[f], Rs[f], tri, 5, 5, f"sparse {band} mutual {mutual} frame {f}")
            if band[0] == 1.0 and not mutual:
                ref = sparse_frame_np(Ls[0], Rs[0], tri, band)
                uv_r, xyz, st = sp.subpixel_refine(Ls[0], Rs[0], ref["uv_l"], ref["uv_r"], ref["status"], 5, 5, tri)
                got = res.frame(0)
                np.testing.assert_array_equal(got["status"], st)
                ok = st == o.ST_OK
                np.testing.assert_array_equal(got["uv_r"][ok], uv_r[ok])
                np.testing.assert_array_equal(got["xyz"][ok], xyz[ok])


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_raw_frames_refine_on_the_rectified_planes(vi_cams):
    """With rectification set, the refinement reads the rectified planes the detector read (svi_rectify gives them)."""
    from svi_mapper_b200.synth import unrectify
    W, H = vi_cams[0].width, vi_cams[0].height
    pairs = [stereo_pair(W, H, 4200 + i) for i in range(3)]
    RL = np.stack([unrectify(p[0], vi_cams[0]) for p in pairs])
    RR = np.stack([unrectify(p[1], vi_cams[1]) for p in pairs])
    tri = _tri(vi_cams)
    with _fe(vi_cams, chunk_frames=2) as off, _fe(vi_cams, chunk_frames=2, subpixel_window=5, subpixel_search=5) as fe:
        off.set_rectification(*vi_cams)
        fe.set_rectification(*vi_cams)
        L, R = fe.rectify(RL, 0), fe.rectify(RR, 1)
        res, base = fe.stereo_frames(RL, RR), off.stereo_frames(RL, RR)
        sres, sbase = fe.stereo_frames_sparse(RL, RR, None, 1.0, 1.0, 60.0), off.stereo_frames_sparse(RL, RR, None, 1.0, 1.0, 60.0)
        for f in range(3):
            n_ok, _, _ = assert_refined(res.frame(f), base.frame(f), L[f], R[f], tri, 5, 5, f"raw dense frame {f}")
            assert n_ok > 100
            assert_refined(sres.frame(f), sbase.frame(f), L[f], R[f], tri, 5, 5, f"raw sparse frame {f}")


def assert_same_results(got, want):
    """Every output svi_stereo_result defines, byte for byte: the per-frame counts, every field of the slots below
    n_keypoints, and uv_right / xyz_left / desc_right of the SVI_OK ones.  The slots behind n_keypoints are unspecified
    after a call (include/svi_gpu.h) and hold whatever the device scratch held, so they are not compared."""
    for k in ("n_keypoints", "n_detected", "n_keypoints_right"):
        if getattr(want, k) is not None:
            np.testing.assert_array_equal(getattr(got, k), getattr(want, k), err_msg=k)
    for f in range(len(want.n_keypoints)):
        g, w = got.frame(f), want.frame(f)
        for k in UNCHANGED + ("status",) + (("second",) if "second" in w else ()):
            np.testing.assert_array_equal(g[k], w[k], err_msg=f"frame {f} {k}")
        ok = w["status"] == o.ST_OK
        for k in ("uv_r", "xyz", "desc_r"):
            np.testing.assert_array_equal(g[k][ok], w[k][ok], err_msg=f"frame {f} {k}")


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_mode_off_parameters_launches_and_stages(kitti_cams):
    """w = 0 (any L) is the default ctx byte for byte; invalid (w, L) are refused by svi_create and w + L = 28 is accepted;
    one more launch per chunk on both paths; the 'subpixel' stage has launches only with the mode on; multi-GPU driver."""
    from svi_mapper_b200 import MultiFrontend, SviError, _lib
    W, H = kitti_cams[0].width, kitti_cams[0].height
    pairs = [stereo_pair(W, H, 60 + i) for i in range(3)]
    Ls, Rs = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    with _fe(kitti_cams) as dflt, _fe(kitti_cams, subpixel_window=0, subpixel_search=99) as zero:
        for call in (lambda fe: fe.stereo_frames(Ls, Rs), lambda fe: fe.stereo_frames(Ls[:1], Rs[:1]),
                     lambda fe: fe.stereo_frames_sparse(Ls, Rs, None, 1.0, 1.0, 60.0, mutual=True)):
            assert_same_results(call(zero), call(dflt))
        k_default = (dflt.kernels_per_chunk(64), dflt.kernels_per_chunk(1))
        assert (zero.kernels_per_chunk(64), zero.kernels_per_chunk(1)) == k_default
        dflt.set_profiling(2)
        dflt.stereo_frames(Ls, Rs)
        assert dflt.stage_timings()["subpixel"]["launches"] == 0
    for w, Lr in ((-1, 5), (5, 0), (5, -2), (20, 9), (1, 28), (28, 1)):
        with pytest.raises(SviError) as e:
            _fe(kitti_cams, subpixel_window=w, subpixel_search=Lr)
        assert e.value.code == _lib.SVI_ERR_INVALID, (w, Lr)
    for w, Lr in ((27, 1), (1, 27), (12, 16)):
        with _fe(kitti_cams, subpixel_window=w, subpixel_search=Lr) as fe:
            assert (fe.kernels_per_chunk(64), fe.kernels_per_chunk(1)) == (k_default[0] + 1, k_default[1] + 1)
            fe.set_profiling(2)
            fe.stereo_frames(Ls, Rs)
            st = fe.stage_timings()["subpixel"]
            assert st["launches"] >= 1 and st["total_ms"] > 0
            if (w, Lr) == (27, 1):   # the widest patches still stay inside the image
                res = fe.stereo_frames(Ls, Rs)
                assert (res.status == _lib.SVI_OK).sum() > 100
    assert _lib.load().svi_status_text(_lib.SVI_SUBPIXEL_REJECTED).decode().startswith("sub-pixel refinement")
    with _fe(kitti_cams, subpixel_window=5, subpixel_search=5) as one, \
            MultiFrontend(*kitti_cams, devices=[0, 0], subpixel_window=5, subpixel_search=5) as multi:
        assert_same_results(multi.stereo_frames(Ls, Rs), one.stereo_frames(Ls, Rs))


@pytest.mark.gpu
def test_bounds_checked_build_subpixel():
    """The dense, masked and sparse parity cases once against the -DSVI_BOUNDS_CHECK build, in which every run-time index of
    subpixel_refine_kernel is asserted and a failed assertion fails the next call."""
    from svi_mapper_b200 import build as bld
    lib = bld.build_checked()
    env = dict(os.environ, SVI_GPU_LIB=str(lib))
    r = subprocess.run([sys.executable, "-m", "pytest", str(pathlib.Path(__file__)), "-x", "-q", "-m", "gpu",
                        "-k", "dense_batch or masked or sparse_frames"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "5 passed" in r.stdout and "failed" not in r.stdout
