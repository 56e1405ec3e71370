"""The left-right (mutual) check of sparse stereo frames (svi_sparse_band.mutual, SVI_SPARSE_NOT_MUTUAL).

A LEFT slot matched to RIGHT key-point j keeps its match only if j's own first arg-min over the frame's LEFT key-points,
under the same admissibility relation, is this slot: cv2.BFMatcher(NORM_HAMMING, crossCheck=True).  Status order: no match,
the cut-off, the check, getPointInLEFT.  The reverse relation is the forward one with the roles swapped and the disparity
bounds mirrored, which fp32 subtraction makes exact; so svi_match_epipolar called twice is an exact composed oracle.

CPU tier: the numpy restatement against cv2's crossCheck (brute force) and two masked BFMatcher calls (narrow bands), ties
in both directions; the precision gain on a seeded pair.  GPU tier: the fused call byte for byte against the restatement
and the composed public calls, check off against check on, edge frames, the device entry, errors, rectification, a C5-sized
frame, and a rerun against the bounds-checked build."""
import os
import pathlib
import subprocess
import sys

import numpy as np
import pytest

from oracle import frontend_np as o
from svi_mapper_b200.synth import disparity_field, stereo_pair
from test_sparse_frames import BANDS, FAST, _fe, _tri, assert_same, composed_np, keypoints_np, sparse_frame_np

F32 = np.float32
ST_SPARSE_NOT_MUTUAL = 25   # svi_status SVI_SPARSE_NOT_MUTUAL


# ------------------------------------------------------------------------------------------------- numpy restatement
def mirrored(band):
    """The reverse pass's band: RIGHT queries, LEFT trains, bounds (-max_disparity, -min_disparity)."""
    return band[0], -F32(band[2]), -F32(band[1])


def mutual_pairs_np(dl, kl, dr, kr, band):
    """First arg-min both ways: (forward index per LEFT key-point, bool per LEFT key-point: the match is mutual)."""
    idx = o.match_epipolar(dl, np.asarray(kl, F32), dr, np.asarray(kr, F32), *band)[0]
    return idx, is_mutual(idx, o.match_epipolar(dr, np.asarray(kr, F32), dl, np.asarray(kl, F32), *mirrored(band))[0])


def is_mutual(idx, rev):
    ok = idx >= 0
    m = np.zeros(len(idx), bool)
    m[ok] = rev[idx[ok]] == np.flatnonzero(ok)
    return m


def apply_mutual(frame: dict, mutual) -> dict:
    """The check on a frame without it: slots past the cut-off whose match is not mutual become SVI_SPARSE_NOT_MUTUAL."""
    out = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in frame.items()}
    st = out["status"]
    rej = (st != o.ST_TRI_NO_MATCH) & (st != o.ST_TRI_DISTANCE) & ~mutual
    st[rej] = ST_SPARSE_NOT_MUTUAL
    for k in ("uv_r", "xyz", "desc_r"):
        out[k][rej] = 0
    return out


def sparse_frame_mutual_np(L, R, tri, band, mask=None, **det) -> dict:
    """sparse_frame_np with the check: forward and mirrored reverse match_epipolar, then the status order."""
    fwd = sparse_frame_np(L, R, tri, band, mask, **det)
    kr, dr = keypoints_np(R, None, **det)
    rev = o.match_epipolar(dr, kr.astype(F32), fwd["desc_l"], fwd["uv_l"], *mirrored(band))[0]
    return apply_mutual(fwd, is_mutual(fwd["idx"], rev))


def composed_mutual(fe, L, R, band, mask=None) -> dict:
    """The same frame through public calls: composed_np, then match_epipolar again with swapped lists and mirrored bounds."""
    fwd = composed_np(fe, L, R, band, mask)
    kr = fe.detect(R)[0]
    dr, keep = fe.describe(R, kr)
    kr, dr = kr[keep], dr[keep]
    rev = fe.match_epipolar(dr, kr, fwd["desc_l"], fwd["uv_l"], *mirrored(band))[0]
    return apply_mutual(fwd, is_mutual(fwd["idx"], rev))


# ------------------------------------------------------------------------------------------------------------ CPU tier
def _cv2():
    cv2 = pytest.importorskip("cv2")
    cv2.setUseOptimized(False)
    cv2.setNumThreads(1)
    return cv2


def _band_mask(kq, kt, band):
    d = kq[:, None, 0].astype(F32) - kt[None, :, 0].astype(F32)
    return ((np.abs(kq[:, None, 1].astype(F32) - kt[None, :, 1].astype(F32)) <= F32(band[0])) & (d >= F32(band[1])) &
            (d <= F32(band[2])))


@pytest.mark.parametrize("name,seed", [("vi_sensor", 11), ("kitti_11_12", 12)])
def test_mutual_restatement_matches_cv2(name, seed):
    """Brute force: the restatement's mutual pairs == BFMatcher(crossCheck=True).match.  Narrow bands (cv2 refuses crossCheck
    with a mask): == two masked BFMatcher.match calls, with mask and mask.T, and the mirrored band's mask is exactly mask.T.
    Ties both ways: duplicated RIGHT descriptors in one LEFT key-point's band, duplicated LEFT descriptors on one row."""
    cv2 = _cv2()
    W, H = (376, 240) if name == "vi_sensor" else (620, 188)
    L, R = stereo_pair(W, H, seed)
    kl, dl = keypoints_np(L)
    kr, dr = keypoints_np(R)
    kl, dl, kr, dr = kl.copy(), dl.copy(), kr.copy(), dr.copy()
    dr[3] = dr[4] = dl[0]                       # RIGHT tie: LEFT 0 sees two equal trains, the lower index wins
    kr[3] = kr[4] = kl[0] - [5, 0]
    dl[7] = dl[8] = dr[10]                      # LEFT tie on one row: RIGHT 10 sees two equal LEFT trains
    kl[8] = kl[7] + [3, 0]
    kr[10] = kl[7] - [6, 0]
    for band in ((1.0, 1.0, 60.0), (0.0, 1.0, 60.0), (3.0, 0.0, 1e9), (1e9, -1e9, 1e9)):
        idx, mutual = mutual_pairs_np(dl, kl, dr, kr, band)
        got = {(i, int(idx[i])) for i in np.flatnonzero(mutual)}
        mask = _band_mask(kl, kr, band)
        np.testing.assert_array_equal(_band_mask(kr, kl, mirrored(band)), mask.T)
        if band[0] >= 1e9:
            ref = {(m.queryIdx, m.trainIdx) for m in cv2.BFMatcher(cv2.NORM_HAMMING, crossCheck=True).match(dl, dr)}
        else:
            bf = cv2.BFMatcher(cv2.NORM_HAMMING)
            back = {m.queryIdx: m.trainIdx for m in bf.match(dr, dl, np.ascontiguousarray(mask.T, np.uint8))}
            ref = {(m.queryIdx, m.trainIdx) for m in bf.match(dl, dr, mask.astype(np.uint8)) if back.get(m.trainIdx) == m.queryIdx}
        assert got == ref, band
        assert len(got) > 10
        if band[0] >= 1:
            assert idx[0] == 3 and (0, 3) in got and not mutual[[7, 8]].all() and (7, 10) in got and (8, 10) not in got


def test_mutual_first_argmin_equals_cv2_crosscheck_on_ties():
    """300 small random cases drawn from a few descriptors (ties everywhere): cv2's crossCheck == first arg-min both ways."""
    cv2 = _cv2()
    rng = np.random.default_rng(5)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING, crossCheck=True)
    for _ in range(300):
        pool = rng.integers(0, 256, (int(rng.integers(2, 6)), 32), dtype=np.uint8)
        pool[1:] = pool[0] ^ (rng.random((len(pool) - 1, 32)) < 0.02).astype(np.uint8)
        dl = pool[rng.integers(0, len(pool), int(rng.integers(1, 25)))]
        dr = pool[rng.integers(0, len(pool), int(rng.integers(1, 25)))]
        kl, kr = np.zeros((len(dl), 2), F32), np.zeros((len(dr), 2), F32)
        idx, mutual = mutual_pairs_np(dl, kl, dr, kr, (1e9, -1e9, 1e9))
        assert {(i, int(idx[i])) for i in np.flatnonzero(mutual)} == {(m.queryIdx, m.trainIdx) for m in bf.match(dl, dr)}


def _precision(kl, kr, idx, dist, accept, d_true):
    """(accepted, correct): correct = same row and |x_L - x_R - d_true(x_R, y)| <= 1."""
    acc = accept & (idx >= 0) & (dist < 100)
    j = idx[acc]
    good = (kr[j, 1] == kl[acc, 1]) & (np.abs(kl[acc, 0] - kr[j, 0] - d_true[kr[j, 1], kr[j, 0]]) <= 1)
    return int(acc.sum()), int(good.sum())


def test_mutual_precision_on_seeded_pair():
    """1241 x 376, seed 7, GFTT: on a brute-force band, under 10 % of the cut-off's matches are right and over 50 % with
    the check; on a +-1 row band precision rises too; the check drops no correct match on either."""
    W, H, seed = 1241, 376, 7
    L, R = stereo_pair(W, H, seed, 1, 55)
    d_true = disparity_field(W, H, np.random.default_rng(seed + 0x5EED), 1, 55)
    kl, dl = keypoints_np(L)
    kr, dr = keypoints_np(R)
    for band, lo, hi in (((1e9, -1e9, 1e9), 0.10, 0.50), ((1.0, 1.0, 60.0), 0.0, 0.0)):
        idx, dist, _ = o.match_epipolar(dl, kl.astype(F32), dr, kr.astype(F32), *band)
        mutual = mutual_pairs_np(dl, kl, dr, kr, band)[1]
        n0, g0 = _precision(kl, kr, idx, dist, np.ones(len(kl), bool), d_true)
        n1, g1 = _precision(kl, kr, idx, dist, mutual, d_true)
        assert g1 == g0 > 50 and n1 < n0, (band, n0, g0, n1, g1)
        assert g1 / n1 > g0 / n0
        if lo:
            assert g0 / n0 < lo and g1 / n1 > hi, (n0, g0, n1, g1)


# ------------------------------------------------------------------------------------------------------------ GPU tier
def _assert_off_on(off, on):
    """mutual=True against mutual=False: equal but for status (OK / zero disparity -> not mutual) and the OK-only fields of
    the slots it rejects."""
    for k in ("n_keypoints", "n_detected", "n_keypoints_right"):
        np.testing.assert_array_equal(getattr(on, k), getattr(off, k))
    for f in range(len(off.n_keypoints)):
        a, b = off.frame(f), on.frame(f)
        for k in ("uv_l", "desc_l", "dist", "idx", "second"):
            np.testing.assert_array_equal(b[k], a[k], err_msg=k)
        ch = a["status"] != b["status"]
        assert (b["status"][ch] == ST_SPARSE_NOT_MUTUAL).all()
        assert np.isin(a["status"][ch], (o.ST_OK, o.ST_TRI_ZERO_DISP)).all()
        ok = b["status"] == o.ST_OK
        for k in ("uv_r", "desc_r", "xyz"):
            np.testing.assert_array_equal(b[k][ok], a[k][ok], err_msg=k)


def _assert_identical(x, y):
    for k, v in vars(x).items():
        np.testing.assert_array_equal(getattr(y, k), v, err_msg=k)


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
@pytest.mark.parametrize("detector", ["gftt", "fast"])
def test_sparse_mutual_equal_oracle_and_composed_calls(kitti_cams, detector):
    """Five frames in chunks of two (three chunks, the last ragged), masks on some frames, the four bands: the check equals
    the composed public calls on every frame and the numpy restatement on a subset; mutual=False is byte-identical to the
    call without the argument, and mutual=True differs from it only in status and the OK-only fields."""
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
        for band in BANDS:
            plain = fe.stereo_frames_sparse(Ls, Rs, masks, *band)
            _assert_identical(plain, fe.stereo_frames_sparse(Ls, Rs, masks, *band, mutual=False))
            res = fe.stereo_frames_sparse(Ls, Rs, masks, *band, mutual=True)
            _assert_off_on(plain, res)
            for f in range(5):
                got = res.frame(f)
                assert_same(got, composed_mutual(fe, Ls[f], Rs[f], band, masks[f]), f"composed {band} frame {f}")
                if f in (0, 3) and band in (BANDS[0], BANDS[3]):   # the numpy restatement is slow: a subset
                    assert_same(got, sparse_frame_mutual_np(Ls[f], Rs[f], tri, band, masks[f], **det), f"oracle {band} frame {f}")
            st = np.concatenate([res.frame(f)["status"] for f in range(5)])
            assert (st == o.ST_OK).sum() > 200 and (st == ST_SPARSE_NOT_MUTUAL).sum() > 0, band


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_sparse_mutual_edge_frames(kitti_cams):
    """Exact reverse ties (a LEFT image of one block repeated side by side: equal LEFT descriptors in one band, the lowest
    slot keeps the match and the others are not mutual), a black RIGHT frame (no reverse queries) and a black LEFT frame
    (no reverse trains), in one batch."""
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
            res = fe.stereo_frames_sparse(Ls, Rs, None, *band, mutual=True)
            _assert_off_on(fe.stereo_frames_sparse(Ls, Rs, None, *band), res)
            f0 = res.frame(0)
            assert_same(f0, sparse_frame_mutual_np(P, PR, tri, band), f"ties {band}")
            assert_same(f0, composed_mutual(fe, P, PR, band), f"ties composed {band}")
            if band[0] >= 1e9:
                # every LEFT copy of a descriptor matches the same RIGHT key-point at distance 0: the lowest slot keeps it
                groups = 0
                for j in np.unique(f0["idx"][f0["dist"] == 0]):
                    s = np.flatnonzero((f0["idx"] == j) & (f0["dist"] == 0))
                    if len(s) > 1:
                        groups += 1
                        assert f0["status"][s[0]] != ST_SPARSE_NOT_MUTUAL
                        assert (f0["status"][s[1:]] == ST_SPARSE_NOT_MUTUAL).all()
                assert groups > 20
            f1 = res.frame(1)
            assert len(f1["uv_l"]) > 100 and f1["n_right"] == 0
            assert (f1["status"] == o.ST_TRI_NO_MATCH).all() and (f1["idx"] == -1).all()
            assert res.n_keypoints[2] == 0 and res.n_keypoints_right[2] > 100


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_sparse_mutual_device_entry_and_errors(kitti_cams):
    """stereo_frames_sparse_device with the check equals the host call; mutual = 2 is SVI_ERR_INVALID on both entries."""
    import torch
    from svi_mapper_b200 import SviError, _lib
    W, H = kitti_cams[0].width, kitti_cams[0].height
    pairs = [stereo_pair(W, H, 900 + i) for i in range(3)]
    Ls, Rs = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    masks = np.full_like(Ls, 255)
    masks[1, 100:200, 300:700] = 0
    keys = ("n_keypoints", "n_detected", "uv_left", "uv_right", "xyz_left", "desc_left", "desc_right", "distance", "match_index", "status")
    with _fe(kitti_cams, chunk_frames=2) as fe:
        dl, dr, dm = (torch.from_numpy(a).cuda() for a in (Ls, Rs, masks))
        for band in (BANDS[0], BANDS[3]):
            want = fe.stereo_frames_sparse(Ls, Rs, masks, *band, mutual=True)
            assert (want.status == ST_SPARSE_NOT_MUTUAL).sum() > 0
            dev = {k: torch.from_numpy(v).cuda().zero_() for k, v in vars(want).items()}
            r = _lib.StereoResult(fe.max_corners, *[dev[k].data_ptr() for k in keys])
            sp = _lib.SparseResult(dev["second_distance"].data_ptr(), dev["n_keypoints_right"].data_ptr())
            stream = torch.cuda.Stream()
            fe.stereo_frames_sparse_device(dl.data_ptr(), dr.data_ptr(), W, W * H, 3, r, sp, *band, masks_ptr=dm.data_ptr(),
                                           stream=stream.cuda_stream, mutual=True)
            stream.synchronize()
            fe.check_overflow()
            got = type(want)(**{k: v.cpu().numpy() for k, v in dev.items()})
            np.testing.assert_array_equal(got.n_keypoints_right, want.n_keypoints_right)
            for f in range(3):
                assert_same(got.frame(f), want.frame(f), f"device {band} frame {f}")
        with pytest.raises(SviError) as e:
            fe.stereo_frames_sparse(Ls[:1], Rs[:1], None, *BANDS[0], mutual=2)
        assert e.value.code == _lib.SVI_ERR_INVALID
        with pytest.raises(SviError) as e:
            fe.stereo_frames_sparse_device(dl.data_ptr(), dr.data_ptr(), W, W * H, 1, r, sp, *BANDS[0], mutual=2)
        assert e.value.code == _lib.SVI_ERR_INVALID
        assert fe.stereo_frames_sparse(Ls[:1], Rs[:1], None, *BANDS[0], mutual=True).n_keypoints[0] > 0   # still usable


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_sparse_mutual_on_raw_images(vi_cams):
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
            got = fe.stereo_frames_sparse(RL, RR, None, *band, mutual=True)
            want = plain.stereo_frames_sparse(L, R, None, *band, mutual=True)
            for f in range(3):
                assert_same(got.frame(f), want.frame(f), f"raw {band} frame {f}")
            assert want.n_keypoints.min() > 100 and (want.status == ST_SPARSE_NOT_MUTUAL).sum() > 0


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_sparse_mutual_c5_frame_brute_force(kitti_cams):
    """C5 size: one 3840 x 1080 pair, ~10 k key-points per side, brute-force band: equals the composed calls."""
    from types import SimpleNamespace
    W, H, K = 3840, 1080, 10000
    cl, cr = (SimpleNamespace(width=W, height=H, P=c.P) for c in kitti_cams)
    L, R = stereo_pair(W, H, 3000, d_max=900)
    with _fe((cl, cr), max_corners=K, search_range_px=1000.0, max_candidates=131072, chunk_frames=1) as fe:
        band = (1e9, -1e9, 1e9)
        got = fe.stereo_frames_sparse(L, R, None, *band, mutual=True).frame(0)
        assert len(got["uv_l"]) > 8000 and got["n_right"] > 1000
        assert (got["status"] == ST_SPARSE_NOT_MUTUAL).sum() > 1000
        assert_same(got, composed_mutual(fe, L, R, band), "C5 brute force")


@pytest.mark.gpu
def test_bounds_checked_build_sparse_mutual():
    """The GPU tests of this file once against the -DSVI_BOUNDS_CHECK build, in which every run-time index of the reverse
    pass, the gather and the check is asserted and a failed assertion fails the next call."""
    from svi_mapper_b200 import build as bld
    lib = bld.build_checked()
    env = dict(os.environ, SVI_GPU_LIB=str(lib))
    r = subprocess.run([sys.executable, "-m", "pytest", str(pathlib.Path(__file__)), "-x", "-q", "-m", "gpu", "-k", "not bounds_checked"],
                       env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "6 passed" in r.stdout and "failed" not in r.stdout
