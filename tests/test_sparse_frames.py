"""Sparse stereo frames (svi_stereo_frames_sparse[_device]): LEFT key-points matched against RIGHT key-points inside an
epipolar row band in one batched call, and svi_match_epipolar on the same band matcher.

CPU tier: the numpy restatement of a sparse frame (below, built from the oracle's gftt, brief32, match_epipolar, the cut-off
and Triangulator.point_in_left) against cv2.  GPU tier: the fused call byte for byte against that restatement, against the
composed public calls it replaces (detect, describe on both images, match_epipolar, the cut-off, point_in_left) and against
stereo_frames for the LEFT fields; the device entry, capacity errors, rectification, a C5-sized frame, and a rerun against the
bounds-checked build."""
import os
import pathlib
import subprocess
import sys

import numpy as np
import pytest

from oracle import frontend_np as o
from svi_mapper_b200.synth import stereo_pair

F32 = np.float32
ROOT = pathlib.Path(__file__).resolve().parents[1]
CALIB = ROOT / "tests" / "golden" / "calib"
BANDS = [(1.0, 1.0, 60.0), (0.0, 1.0, 60.0), (3.0, 0.0, 1e9), (1e9, -1e9, 1e9)]   # the last one: brute force
FAST = dict(detector=1, fast_threshold=20, fast_nonmax=1, max_corners=20000, max_candidates=65536)


def _cams(name):
    from svi_mapper_b200 import load_camera
    return load_camera(str(CALIB / f"{name}_left.txt")), load_camera(str(CALIB / f"{name}_right.txt"))


def _tri(cams, **kw):
    cl, cr = cams
    return o.Triangulator(o.Camera(cl.width, cl.height, cl.P), o.Camera(cr.width, cr.height, cr.P), o.StereoParams(**kw))


# ------------------------------------------------------------------------------------------------- numpy restatement
def keypoints_np(img, mask=None, max_corners=1000, detector=0, fast_threshold=20, fast_nonmax=1):
    """The detector of the ctx, then BRIEF's border filter: (xy (k, 2) int32, desc (k, 32) u8) in detector order."""
    xy = o.gftt(img, max_corners, mask=mask) if detector == 0 else o.fast9_16(img, fast_threshold, bool(fast_nonmax))[0]
    if detector == 1 and mask is not None:
        xy = xy[mask[xy[:, 1], xy[:, 0]] != 0]
    keep, desc = o.brief32(img, xy.astype(F32))
    return (xy[keep] if len(keep) else xy[:0]), desc


def sparse_frame_np(L, R, tri: o.Triangulator, band, mask=None, **det) -> dict:
    """One sparse frame: per LEFT key-point the first arg-min over the admissible RIGHT key-points, the second-smallest
    distance, the cut-off (!(distance < match_cutoff)) and getPointInLEFT."""
    kl, dl = keypoints_np(L, mask, **det)
    kr, dr = keypoints_np(R, None, **det)
    n = len(kl)
    idx, dist, second = o.match_epipolar(dl, kl.astype(F32), dr, kr.astype(F32), *band)
    out = dict(uv_l=kl.astype(F32), desc_l=dl, idx=idx, dist=dist, second=second, status=np.zeros(n, np.uint8),
               uv_r=np.zeros((n, 2), F32), xyz=np.zeros((n, 3)), desc_r=np.zeros((n, 32), np.uint8), n_right=len(kr))
    for i in range(n):
        if idx[i] < 0:
            out["status"][i] = o.ST_TRI_NO_MATCH
        elif not (F32(dist[i]) < F32(tri.p.match_cutoff)):
            out["status"][i] = o.ST_TRI_DISTANCE
        else:
            st, xyz = tri.point_in_left(kl[i].astype(F32), kr[idx[i]].astype(F32))
            out["status"][i] = st
            if st == o.ST_OK:
                out["uv_r"][i], out["xyz"][i], out["desc_r"][i] = kr[idx[i]], xyz, dr[idx[i]]
    return out


def composed_np(fe, L, R, band, mask=None) -> dict:
    """The same frame through the composed public calls the fused one replaces."""
    kl = fe.detect(L, mask)[0]
    dl, keep_l = fe.describe(L, kl)
    kr = fe.detect(R)[0]
    dr, keep_r = fe.describe(R, kr)
    kl, dl, kr, dr = kl[keep_l], dl[keep_l], kr[keep_r], dr[keep_r]
    idx, dist, second = fe.match_epipolar(dl, kl, dr, kr, *band)
    n = len(kl)
    status = np.full(n, o.ST_TRI_NO_MATCH, np.uint8)
    status[(idx >= 0) & ~(dist.astype(F32) < F32(fe.params.match_cutoff))] = o.ST_TRI_DISTANCE
    cand = (idx >= 0) & (dist.astype(F32) < F32(fe.params.match_cutoff))
    uv_r = np.zeros((n, 2), F32)
    uv_r[idx >= 0] = kr[idx[idx >= 0]]
    xyz, st = fe.point_in_left(kl, uv_r) if n else (np.zeros((0, 3)), np.zeros(0, np.uint8))
    status[cand] = st[cand]
    ok = status == o.ST_OK
    desc_r = np.zeros((n, 32), np.uint8)
    desc_r[ok] = dr[idx[ok]]
    return dict(uv_l=kl, desc_l=dl, idx=idx, dist=dist, second=second, status=status, uv_r=np.where(ok[:, None], uv_r, 0),
                xyz=np.where(ok[:, None], xyz, 0), desc_r=desc_r, n_right=len(kr))


def assert_same(got: dict, ref: dict, what=""):
    assert len(got["uv_l"]) == len(ref["uv_l"]), what
    assert got["n_right"] == ref["n_right"], what
    for k in ("uv_l", "desc_l", "idx", "dist", "second", "status"):
        np.testing.assert_array_equal(got[k], ref[k], err_msg=f"{what} {k}")
    ok = ref["status"] == o.ST_OK
    for k in ("uv_r", "desc_r", "xyz"):
        np.testing.assert_array_equal(got[k][ok], ref[k][ok], err_msg=f"{what} {k}")


# ------------------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("name,seed", [("vi_sensor", 11), ("kitti_11_12", 12)])
def test_sparse_restatement_matches_cv2(name, seed):
    """The restatement's pieces against cv2 on small vi_sensor- and KITTI-shaped pairs: detection == goodFeaturesToTrack,
    index and distance == BFMatcher.match(q, t, band mask), second distance == knnMatch(k=2, band mask); with constructed
    ties (duplicated RIGHT descriptors in the band) and empty bands."""
    cv2 = pytest.importorskip("cv2")
    cv2.setUseOptimized(False)
    cv2.setNumThreads(1)
    W, H = (376, 240) if name == "vi_sensor" else (620, 188)
    L, R = stereo_pair(W, H, seed)
    for img in (L, R):
        ref = cv2.goodFeaturesToTrack(img, 1000, 0.01, 7.0, blockSize=7, useHarrisDetector=True, k=0.04)
        np.testing.assert_array_equal(o.gftt(img, 1000), ref.reshape(-1, 2).astype(np.int32))
    kl, dl = keypoints_np(L)
    kr, dr = keypoints_np(R)
    dr = dr.copy()
    kr = kr.copy()
    dr[3] = dr[4] = dl[0]            # a tie inside the band of query 0: the lower index wins
    kr[3] = kr[4] = kl[0] - [5, 0]
    for band in ((1.0, 1.0, 60.0), (0.0, 1.0, 60.0), (3.0, 0.0, 1e9), (-1.0, 0.0, 1e9)):
        idx, dist, second = o.match_epipolar(dl, kl.astype(F32), dr, kr.astype(F32), *band)
        d = kl[:, None, 0].astype(F32) - kr[None, :, 0].astype(F32)
        mask = ((np.abs(kl[:, None, 1].astype(F32) - kr[None, :, 1].astype(F32)) <= F32(band[0])) & (d >= F32(band[1])) &
                (d <= F32(band[2]))).astype(np.uint8)
        bf = cv2.BFMatcher(cv2.NORM_HAMMING)
        got = {m.queryIdx: (m.trainIdx, int(m.distance)) for m in bf.match(dl, dr, mask)}
        knn = {ms[0].queryIdx: ms for ms in bf.knnMatch(dl, dr, k=2, mask=mask) if ms}
        for i in range(len(kl)):
            if idx[i] < 0:
                assert i not in got and second[i] == -1
                continue
            assert got[i] == (idx[i], dist[i])
            assert second[i] == (int(knn[i][1].distance) if len(knn[i]) > 1 else -1)
        if band[0] >= 1:
            assert idx[0] == 3 and dist[0] == 0 and second[0] == 0
        if band[0] < 0:
            assert (idx == -1).all()
        else:
            assert (idx >= 0).sum() > 20


# ------------------------------------------------------------------------------------------------------------ GPU tier
def _fe(cams, **kw):
    from svi_mapper_b200 import StereoFrontend
    return StereoFrontend(*cams, **kw)


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
@pytest.mark.parametrize("detector", ["gftt", "fast"])
def test_sparse_frames_equal_oracle_and_composed_calls(kitti_cams, detector):
    """Five frames in chunks of two (three chunks on three lanes, the last one ragged), masks on some frames, four bands:
    every frame equals the numpy restatement and the composed calls; the LEFT fields equal stereo_frames'."""
    W, H = kitti_cams[0].width, kitti_cams[0].height
    pairs = [stereo_pair(W, H, 500 + i) for i in range(5)]
    Ls, Rs = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    rng = np.random.default_rng(8)
    masks = np.stack([o.mask_active_landmarks(W, H, np.stack([rng.uniform(0, W, 150 * (i % 2)), rng.uniform(0, H, 150 * (i % 2))], 1))
                      for i in range(5)])
    kw = dict(FAST) if detector == "fast" else {}
    det = dict(max_corners=kw.get("max_corners", 1000), detector=kw.get("detector", 0))
    tri = _tri(kitti_cams)
    with _fe(kitti_cams, chunk_frames=2, **kw) as fe:
        dense = fe.stereo_frames(Ls, Rs, masks)
        for band in BANDS:
            res = fe.stereo_frames_sparse(Ls, Rs, masks, *band)
            np.testing.assert_array_equal(res.n_keypoints, dense.n_keypoints)
            np.testing.assert_array_equal(res.n_detected, dense.n_detected)
            for f in range(5):
                got, d = res.frame(f), dense.frame(f)
                np.testing.assert_array_equal(got["uv_l"], d["uv_l"])
                np.testing.assert_array_equal(got["desc_l"], d["desc_l"])
                assert_same(got, composed_np(fe, Ls[f], Rs[f], band, masks[f]), f"composed {band} frame {f}")
                if f in (0, 3) or band == BANDS[0]:   # the numpy restatement is slow: a subset of the frames
                    assert_same(got, sparse_frame_np(Ls[f], Rs[f], tri, band, masks[f], **det), f"oracle {band} frame {f}")
            if band == BANDS[0]:
                st = np.concatenate([res.frame(f)["status"] for f in range(5)])
                assert (st == 0).sum() > 500 and (st == o.ST_TRI_NO_MATCH).sum() > 0


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_sparse_edge_frames(kitti_cams):
    """Ties (a horizontally periodic texture: equal descriptors in one band), a black RIGHT frame (every slot
    SVI_TRI_NO_MATCH with -1 distances) and a black LEFT frame (no key-points), in one batch."""
    W, H = kitti_cams[0].width, kitti_cams[0].height
    block = stereo_pair(64, H, 77)[0]
    P = np.tile(block, (1, W // 64 + 1))[:, :W]          # period 64: every corner repeats 64 px further right
    PR = np.roll(P, -9, axis=1)
    L, R = stereo_pair(W, H, 78)
    Ls = np.stack([P, L, np.zeros_like(L)])
    Rs = np.stack([PR, np.zeros_like(R), R])
    tri = _tri(kitti_cams)
    with _fe(kitti_cams, chunk_frames=2) as fe:
        for band in ((1.0, 1.0, 200.0), (1e9, -1e9, 1e9)):
            res = fe.stereo_frames_sparse(Ls, Rs, None, *band)
            f0 = res.frame(0)
            assert_same(f0, sparse_frame_np(P, PR, tri, band), f"ties {band}")
            assert_same(f0, composed_np(fe, P, PR, band), f"ties composed {band}")
            assert (f0["second"] == f0["dist"]).sum() > 50      # ties really happened
            f1 = res.frame(1)
            assert len(f1["uv_l"]) > 100 and f1["n_right"] == 0
            assert (f1["status"] == o.ST_TRI_NO_MATCH).all()
            assert (f1["dist"] == -1).all() and (f1["idx"] == -1).all() and (f1["second"] == -1).all()
            assert res.n_keypoints[2] == 0 and res.n_detected[2] == 0 and res.n_keypoints_right[2] > 100


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_sparse_device_entry_and_capacity(kitti_cams):
    """stereo_frames_sparse_device on device tensors equals the host call; a FAST frame with more corners than max_corners on
    RIGHT only is SVI_ERR_CAPACITY from both entry points; bad bands are refused."""
    import torch
    from svi_mapper_b200 import SviError, _lib
    W, H = kitti_cams[0].width, kitti_cams[0].height
    pairs = [stereo_pair(W, H, 900 + i) for i in range(3)]
    Ls, Rs = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    masks = np.full_like(Ls, 255)
    masks[1, 100:200, 300:700] = 0
    with _fe(kitti_cams, chunk_frames=2) as fe:
        for band in (BANDS[0], BANDS[3]):
            want = fe.stereo_frames_sparse(Ls, Rs, masks, *band)
            dev = {k: torch.from_numpy(v).cuda() for k, v in vars(want).items()}
            for v in dev.values():
                v.zero_()
            dl, dr, dm = (torch.from_numpy(a).cuda() for a in (Ls, Rs, masks))
            r = _lib.StereoResult(fe.max_corners, *[dev[k].data_ptr() for k in ("n_keypoints", "n_detected", "uv_left", "uv_right", "xyz_left",
                                                                                 "desc_left", "desc_right", "distance", "match_index", "status")])
            sp = _lib.SparseResult(dev["second_distance"].data_ptr(), dev["n_keypoints_right"].data_ptr())
            stream = torch.cuda.Stream()
            fe.stereo_frames_sparse_device(dl.data_ptr(), dr.data_ptr(), W, W * H, 3, r, sp, *band, masks_ptr=dm.data_ptr(),
                                           stream=stream.cuda_stream)
            stream.synchronize()
            fe.check_overflow()
            got = type(want)(**{k: v.cpu().numpy() for k, v in dev.items()})
            np.testing.assert_array_equal(got.n_keypoints_right, want.n_keypoints_right)
            for f in range(3):
                g, w = got.frame(f), want.frame(f)
                for k in ("uv_l", "desc_l", "idx", "dist", "second", "status"):
                    np.testing.assert_array_equal(g[k], w[k])
                ok = w["status"] == 0
                for k in ("uv_r", "desc_r", "xyz"):
                    np.testing.assert_array_equal(g[k][ok], w[k][ok])
        for bad in ((float("nan"), 0.0, 1.0), (1.0, float("nan"), 1.0), (1.0, 2.0, 1.0)):
            with pytest.raises(SviError) as e:
                fe.stereo_frames_sparse(Ls[:1], Rs[:1], None, *bad)
            assert e.value.code == _lib.SVI_ERR_INVALID
    # FAST: a smooth LEFT image with few corners, a noisy RIGHT one with far more than max_corners
    smooth = np.tile(np.linspace(0, 255, W).astype(np.uint8), (H, 1))
    smooth[100:140, 300:340] = 255
    noisy = np.random.default_rng(3).integers(0, 256, (H, W), dtype=np.uint8)
    with _fe(kitti_cams, detector=1, fast_threshold=20, max_corners=2000, max_candidates=65536) as fe:
        with pytest.raises(SviError) as e:
            fe.stereo_frames_sparse(smooth, noisy)
        assert e.value.code == _lib.SVI_ERR_CAPACITY
        assert len(fe.detect(smooth)[0]) < 2000
        out = fe.stereo_frames_sparse(smooth, smooth)     # the condition was cleared
        assert out.n_keypoints[0] > 0
        res = type(out).empty(1, fe.max_corners, sparse=True)
        dev = {k: torch.from_numpy(v).cuda() for k, v in vars(res).items()}
        r = _lib.StereoResult(fe.max_corners, *[dev[k].data_ptr() for k in ("n_keypoints", "n_detected", "uv_left", "uv_right", "xyz_left",
                                                                             "desc_left", "desc_right", "distance", "match_index", "status")])
        sp = _lib.SparseResult(dev["second_distance"].data_ptr(), dev["n_keypoints_right"].data_ptr())
        dl, dr = torch.from_numpy(smooth).cuda(), torch.from_numpy(noisy).cuda()
        fe.stereo_frames_sparse_device(dl.data_ptr(), dr.data_ptr(), W, W * H, 1, r, sp)
        with pytest.raises(SviError) as e:
            fe.check_overflow()
        assert e.value.code == _lib.SVI_ERR_CAPACITY


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_sparse_frames_on_raw_images(vi_cams):
    """With rectification set, raw frames give the result cv2-rectified frames give without it."""
    import cv2
    from svi_mapper_b200.synth import unrectify
    cv2.setUseOptimized(False)
    cv2.setNumThreads(1)
    W, H = vi_cams[0].width, vi_cams[0].height
    pairs = [stereo_pair(W, H, 4100 + i) for i in range(3)]
    RL = np.stack([unrectify(p[0], vi_cams[0]) for p in pairs])
    RR = np.stack([unrectify(p[1], vi_cams[1]) for p in pairs])

    def rect(cam, raw):
        m1, m2 = cv2.initUndistortRectifyMap(cam.K, cam.distortion, cam.rectification, cam.P, (cam.width, cam.height), cv2.CV_16SC2)
        return np.stack([cv2.remap(r, m1, m2, cv2.INTER_LINEAR) for r in raw])
    L, R = rect(vi_cams[0], RL), rect(vi_cams[1], RR)
    with _fe(vi_cams, chunk_frames=2) as plain, _fe(vi_cams, chunk_frames=2) as fe:
        fe.set_rectification(*vi_cams)
        for band in (BANDS[0], BANDS[3]):
            got, want = fe.stereo_frames_sparse(RL, RR, None, *band), plain.stereo_frames_sparse(L, R, None, *band)
            for f in range(3):
                assert_same(got.frame(f), want.frame(f), f"raw {band} frame {f}")
            assert want.n_keypoints.min() > 100


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_sparse_c5_frame_brute_force(kitti_cams):
    """C5 size: one 3840 x 1080 pair, ~10 k key-points per side, brute-force band: equals the composed calls."""
    from types import SimpleNamespace
    W, H, K = 3840, 1080, 10000
    cl, cr = (SimpleNamespace(width=W, height=H, P=c.P) for c in kitti_cams)
    L, R = stereo_pair(W, H, 3000, d_max=900)
    with _fe((cl, cr), max_corners=K, search_range_px=1000.0, max_candidates=131072, chunk_frames=1) as fe:
        band = (1e9, -1e9, 1e9)
        res = fe.stereo_frames_sparse(L, R, None, *band)
        got = res.frame(0)
        assert len(got["uv_l"]) > 8000 and got["n_right"] > 1000
        assert_same(got, composed_np(fe, L, R, band), "C5 brute force")


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_match_epipolar_float_coordinates(kitti_cams):
    """svi_match_epipolar on the band matcher: fractional coordinates on the band and disparity edges, NaN coordinates
    (never admissible), several CTAs and tiles, an empty train list -- equal to the oracle."""
    rng = np.random.default_rng(6)
    nq, nt = 300, 1100
    q = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    t = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
    t[:200] = q[:200] ^ (rng.random((200, 32)) < 0.05).astype(np.uint8)
    t[200:260] = t[:60]                                                    # exact duplicates: ties
    qxy = np.stack([rng.uniform(50, 900, nq), rng.uniform(0, 40, nq)], 1).astype(F32)
    txy = np.stack([rng.uniform(0, 900, nt), rng.uniform(0, 40, nt)], 1).astype(F32)
    band, dmin, dmax = F32(1.25), F32(0.5), F32(60.75)
    for i in range(100):                                                     # trains exactly on the edges
        j = i % nq
        txy[300 + i] = [qxy[j, 0] - (dmin if i % 4 == 0 else dmax if i % 4 == 1 else 1.0),
                        qxy[j, 1] + (band if i % 3 == 0 else -band if i % 3 == 1 else 0.0)]
    txy[200:260] = txy[:60]
    qxy[5] = [np.nan, 10.0]
    qxy[6] = [100.0, np.nan]
    txy[7] = [np.nan, 3.0]
    txy[8] = [40.0, np.nan]
    with _fe(kitti_cams) as fe:
        for b in ((band, dmin, dmax), (F32(0.0), F32(0.0), F32(1e9)), (F32(1e9), F32(-1e9), F32(1e9))):
            gi, gd, gs = fe.match_epipolar(q, qxy, t, txy, *b)
            ri, rd, rs = o.match_epipolar(q, qxy, t, txy, *b)
            np.testing.assert_array_equal(gi, ri)
            np.testing.assert_array_equal(gd, rd)
            np.testing.assert_array_equal(gs, rs)
            assert gi[5] == -1 and gi[6] == -1 and 7 not in gi and 8 not in gi
        gi, gd, gs = fe.match_epipolar(q[:3], qxy[:3], np.zeros((0, 32), np.uint8), np.zeros((0, 2), F32))
        assert (gi == -1).all() and (gd == -1).all() and (gs == -1).all()


@pytest.mark.gpu
def test_bounds_checked_build_sparse_frames():
    """The GPU tests of this file once against the -DSVI_BOUNDS_CHECK build, in which every run-time index of
    band_match_kernel is asserted and a failed assertion fails the next call."""
    from svi_mapper_b200 import build as bld
    lib = bld.build_checked()
    env = dict(os.environ, SVI_GPU_LIB=str(lib))
    r = subprocess.run([sys.executable, "-m", "pytest", str(pathlib.Path(__file__)), "-x", "-q", "-m", "gpu", "-k", "not bounds_checked"],
                       env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "7 passed" in r.stdout and "failed" not in r.stdout
