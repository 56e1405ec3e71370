"""Left-right consistency check of the dense scan-line matches (svi_params.lr_max_diff), on the device.

CPU tier: the CPU restatement (tests/lr_check_np.py: the oracle's addNewLandmarks, then the reference's reverse search
getPointTriangulatedInLEFT from every SVI_OK match) removes most wrong matches of a KITTI-shaped pair with a known disparity
field and few right ones, and follows each branch of the rule on hand-built rows.  GPU tier: with the check on, every dense
entry point equals the restatement applied to the same call with the check off, byte for byte (status only changes), and
equals the composed public calls (the check off, then svi_triangulate_left on the SVI_OK slots); the check off is the
default ctx; sparse frames ignore it; values below -1 are refused; a rerun against the bounds-checked build."""
import os
import pathlib
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import frontend_np as o
import lr_check_np as lr
import subpixel_np as sp
from svi_mapper_b200.synth import disparity_field, left_image, stereo_pair

F32 = np.float32
TOLS = [0, 1, 3]


def _tri(cams, **kw):
    cl, cr = cams
    return o.Triangulator(o.Camera(cl.width, cl.height, np.asarray(cl.P, np.float64).reshape(3, 4)),
                          o.Camera(cr.width, cr.height, np.asarray(cr.P, np.float64).reshape(3, 4)), o.StereoParams(**kw))


def _sized(cams, W, H):
    return tuple(SimpleNamespace(width=W, height=H, P=c.P) for c in cams)


# ------------------------------------------------------------------------------------------------------------ CPU tier
def test_restatement_removes_wrong_matches_of_a_known_disparity_field(kitti_cams):
    """synth.stereo_pair(1241, 376, seed 7) with the kitti_00 cameras: tolerance 1 rejects at least half of the SVI_OK
    matches whose disparity is more than 1 px off the generator's field and at most 2 % of the others."""
    W, H = kitti_cams[0].width, kitti_cams[0].height
    L, R = stereo_pair(W, H, 7)
    d_true = disparity_field(W, H, np.random.default_rng(7 + 0x5EED))   # synth.right_image's field, on the RIGHT grid
    tri = _tri(kitti_cams)
    base = o.add_new_landmarks(L, R, tri)
    ok = base["status"] == o.ST_OK
    xr, y = base["uv_r"][:, 0].astype(int), base["uv_l"][:, 1].astype(int)
    wrong = ok & (np.abs((base["uv_l"][:, 0] - base["uv_r"][:, 0]) - d_true[y, np.clip(xr, 0, W - 1)]) > 1)
    assert ok.sum() > 700 and wrong.sum() > 50, (ok.sum(), wrong.sum())
    st = lr.lr_check(L, base["uv_l"], base["uv_r"], base["desc_r"], base["status"], 1, tri)
    rej = st == lr.ST_LR_INCONSISTENT
    assert ((st == o.ST_OK) | rej)[ok].all() and (st[~ok] == base["status"][~ok]).all()
    assert (rej & wrong).sum() >= 0.5 * wrong.sum(), ((rej & wrong).sum(), wrong.sum())
    assert (rej & ok & ~wrong).sum() <= 0.02 * (ok & ~wrong).sum(), ((rej & ok & ~wrong).sum(), (ok & ~wrong).sum())
    # the tolerance only loosens the rule
    st0 = lr.lr_check(L, base["uv_l"], base["uv_r"], base["desc_r"], base["status"], 0, tri)
    assert (rej <= (st0 == lr.ST_LR_INCONSISTENT)).all()


def _rows(W=200, H=100, seed=11, period=None):
    rng = np.random.default_rng(seed)
    img = left_image(W, H, seed) if period is None else np.tile(rng.integers(0, 256, (H, period), dtype=np.uint8), (1, W // period + 1))[:, :W]
    return np.ascontiguousarray(img)


def test_restatement_branches_on_hand_built_rows(vi_cams):
    """Each branch of the rule on one LEFT row whose descriptors are known: the RIGHT descriptor is LEFT's at x0, so the
    reverse search from xR lands at x0.  Tolerance 0 rejects a LEFT key-point 1 px away from x0 and tolerance 1 keeps it;
    on columns of period 8 exact reverse ties take the first arg-min (the one nearest xR + 1); a reverse search that lands
    closer to xR than a raised min_disparity_px fails through getPointInLEFT whatever the tolerance."""
    W, H, y, xr = 200, 100, 50, 40
    tri = _tri(_sized(vi_cams, W, H))
    img = _rows(W, H)
    x0 = 70
    _, desc = o.brief32(img, np.array([[x0, y]], F32))
    r = lr.reverse_search(img, (F32(x0), F32(y)), (F32(xr), F32(y)), desc[0], tri)
    assert r["status"] == o.ST_OK and r["uv"][0] == F32(x0) and r["dist"] == 0
    for xl, want0, want1 in ((x0, o.ST_OK, o.ST_OK), (x0 + 1, lr.ST_LR_INCONSISTENT, o.ST_OK), (x0 - 1, lr.ST_LR_INCONSISTENT, o.ST_OK),
                             (x0 + 2, lr.ST_LR_INCONSISTENT, lr.ST_LR_INCONSISTENT)):
        args = (img, [[xl, y]], [[xr, y]], desc, [o.ST_OK])
        assert lr.lr_check(*args, 0, tri)[0] == want0, xl
        assert lr.lr_check(*args, 1, tri)[0] == want1, xl
    # ties: every 8th column holds the same descriptor; the pool starts at xr + 1 = 41, so 48 is the first arg-min
    per = _rows(W, H, 12, period=8)
    _, dp = o.brief32(per, np.array([[64, y]], F32))
    r = lr.reverse_search(per, (F32(64), F32(y)), (F32(xr), F32(y)), dp[0], tri)
    assert r["status"] == o.ST_OK and r["uv"][0] == F32(48) and r["dist"] == 0
    assert lr.lr_check(per, [[48, y], [56, y], [64, y]], [[xr, y]] * 3, np.repeat(dp, 3, 0), [o.ST_OK] * 3, 1, tri).tolist() == \
        [o.ST_OK, lr.ST_LR_INCONSISTENT, lr.ST_LR_INCONSISTENT]
    assert lr.lr_check(per, [[64, y]], [[xr, y]], dp, [o.ST_OK], 15, tri)[0] == lr.ST_LR_INCONSISTENT   # 16 px away
    assert lr.lr_check(per, [[64, y]], [[xr, y]], dp, [o.ST_OK], 16, tri)[0] == o.ST_OK
    # a raised min_disparity_px: the reverse search lands at x0 = xr + 2 (disparity 2), the LEFT key-point is at xr + 6
    _, d2 = o.brief32(img, np.array([[xr + 2, y]], F32))
    args = (img, [[xr + 6, y]], [[xr, y]], d2, [o.ST_OK], 10)
    assert lr.lr_check(*args, tri)[0] == o.ST_OK
    tri5 = _tri(_sized(vi_cams, W, H), min_disparity=5.0)
    assert lr.reverse_search(img, (F32(xr + 6), F32(y)), (F32(xr), F32(y)), d2[0], tri5)["status"] == o.ST_TRI_ZERO_DISP
    assert lr.lr_check(*args, tri5)[0] == lr.ST_LR_INCONSISTENT
    # slots that are not SVI_OK are left alone
    st = lr.lr_check(img, [[x0 + 5, y]] * 3, [[xr, y]] * 3, np.repeat(desc, 3, 0), [o.ST_TRI_DISTANCE, o.ST_TRI_ZERO_DISP, o.ST_TRI_RANGE], 0, tri)
    assert st.tolist() == [o.ST_TRI_DISTANCE, o.ST_TRI_ZERO_DISP, o.ST_TRI_RANGE]


# ------------------------------------------------------------------------------------------------------------ GPU tier
def _fe(cams, **kw):
    from svi_mapper_b200 import StereoFrontend
    return StereoFrontend(*cams, **kw)


LIVE = ("uv_l", "desc_l", "dist", "idx")
OK_ONLY = ("uv_r", "xyz", "desc_r")


def composed(fe_off, off: dict, L, t, size=7.0, search=60.0):
    """The status the check must give, from public calls: `off` (stereo_frames with the check off), then
    svi_triangulate_left on its SVI_OK slots with the RIGHT match and descriptor."""
    st = off["status"].copy()
    ok = np.nonzero(st == o.ST_OK)[0]
    if len(ok) == 0:
        return st
    uv_l, uv_r, half = off["uv_l"][ok], off["uv_r"][ok], F32(4) * F32(size)
    tl = np.stack([uv_r[:, 0] - half, uv_l[:, 1] - half], 1)
    r = fe_off.triangulate_left(L, np.full(len(ok), search, F32), tl, np.stack([uv_r[:, 0], uv_l[:, 1]], 1), off["desc_r"][ok], size)
    keep = (r["status"] == o.ST_OK) & (np.abs(r["uv"][:, 0] - uv_l[:, 0]) <= F32(t))
    st[ok[~keep]] = lr.ST_LR_INCONSISTENT
    return st


def assert_checked(on: dict, off: dict, L, tri, t, what="", fe_off=None, size=7.0, search=60.0, every=1):
    """`on` (check on) == `off` (check off, same call) in every output but status, and status == the restatement's check of
    `off` on every `every`-th slot (and, with fe_off, the composed public calls on every slot)."""
    assert len(on["uv_l"]) == len(off["uv_l"]), what
    for k in LIVE:
        np.testing.assert_array_equal(on[k], off[k], err_msg=f"{what} {k}")
    ok = off["status"] == o.ST_OK
    for k in OK_ONLY:
        np.testing.assert_array_equal(on[k][ok], off[k][ok], err_msg=f"{what} {k}")
    sub = slice(None, None, every)
    st = lr.lr_check(L, off["uv_l"][sub], off["uv_r"][sub], off["desc_r"][sub], off["status"][sub], t, tri, size)
    np.testing.assert_array_equal(on["status"][sub], st, err_msg=f"{what} status")
    if fe_off is not None:
        np.testing.assert_array_equal(composed(fe_off, off, L, t, size, search), on["status"], err_msg=f"{what} composed")
    return int(ok.sum()), int((on["status"] == lr.ST_LR_INCONSISTENT).sum())


def _batch(W, H, n, seed):
    pairs = [stereo_pair(W, H, seed + i) for i in range(n)]
    return np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
@pytest.mark.parametrize("shape", ["kitti_00_binned", "kitti_11_12_per_keypoint", "vi_sensor", "tile_boundary"])
def test_dense_batch_equals_restatement(monkeypatch, kitti_cams, kitti1112_cams, vi_cams, shape):
    """Batches of 26 frames in one chunk (the batch path) at tolerances 0, 1 and 3: kitti_00 with the binned matcher,
    kitti_11_12 with the per-key-point matcher, vi_sensor, and 1241 x 377 (odd height past the Harris stride); one more
    launch per chunk; frame 0 also end to end against the oracle's addNewLandmarks and the check."""
    monkeypatch.setenv("SVI_MATCH_BINNED", "2" if shape == "kitti_00_binned" else "0" if shape == "kitti_11_12_per_keypoint" else "1")
    cams = {"kitti_00_binned": kitti_cams, "kitti_11_12_per_keypoint": kitti1112_cams, "vi_sensor": vi_cams,
            "tile_boundary": _sized(kitti_cams, 1241, 377)}[shape]
    mc = 2000 if shape == "kitti_00_binned" else 1000
    W, H = cams[0].width, cams[0].height
    Ls, Rs = _batch(W, H, 26, 7100)
    tri = _tri(cams, max_corners=mc)
    with _fe(cams, max_corners=mc, chunk_frames=26) as off:
        k_off = off.kernels_per_chunk(26)
        base = off.stereo_frames(Ls, Rs)
        for t in TOLS:
            with _fe(cams, max_corners=mc, chunk_frames=26, lr_max_diff=t) as fe:
                assert fe.kernels_per_chunk(26) == k_off + 1
                res = fe.stereo_frames(Ls, Rs)
                np.testing.assert_array_equal(res.n_keypoints, base.n_keypoints)
                np.testing.assert_array_equal(res.n_detected, base.n_detected)
                for f in (0, 13, 25):
                    n_ok, n_rej = assert_checked(res.frame(f), base.frame(f), Ls[f], tri, t, f"{shape} t={t} frame {f}",
                                                 fe_off=off if f == 13 else None)
                    assert n_ok > 300 and 0 < n_rej < 0.5 * n_ok, (n_ok, n_rej)
                for f in range(26):
                    got, ref = res.frame(f), base.frame(f)
                    changed = got["status"] != ref["status"]
                    assert (ref["status"][changed] == o.ST_OK).all() and (got["status"][changed] == lr.ST_LR_INCONSISTENT).all()
                if t == 1:
                    want = lr.add_new_landmarks(Ls[0], Rs[0], tri, lr_max_diff=1)
                    got = res.frame(0)
                    for k in LIVE + ("status",):
                        np.testing.assert_array_equal(got[k], want[k], err_msg=k)


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_fast_detector(kitti_cams):
    """FAST-9/16 key-points, three frames in chunks of two, tolerance 1."""
    W, H = kitti_cams[0].width, kitti_cams[0].height
    Ls, Rs = _batch(W, H, 3, 7300)
    kw = dict(detector=1, fast_threshold=30, max_corners=60000, max_candidates=65536, chunk_frames=2)
    tri = _tri(kitti_cams)
    with _fe(kitti_cams, **kw) as off, _fe(kitti_cams, lr_max_diff=1, **kw) as fe:
        res, base = fe.stereo_frames(Ls, Rs), off.stereo_frames(Ls, Rs)
        for f in range(3):
            n_ok, n_rej = assert_checked(res.frame(f), base.frame(f), Ls[f], tri, 1, f"FAST frame {f}", fe_off=off, every=1 if f == 0 else 4)
            assert n_ok > 500 and n_rej > 0


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_ragged_masked_batch_device_and_one_pair(kitti_cams, vi_cams):
    """Seven masked frames in chunks of three (3 + 3 + 1); the device entry equals the host entry; the one-pair masked call
    (mask built from landmark centres) equals the oracle's addNewLandmarks followed by the check, end to end."""
    import torch
    from svi_mapper_b200 import _lib
    W, H = kitti_cams[0].width, kitti_cams[0].height
    n, cap = 7, 1000
    Ls, Rs = _batch(W, H, n, 7400)
    rng = np.random.default_rng(5)
    Ms = np.stack([o.mask_active_landmarks(W, H, rng.uniform([0, 0], [W, H], (150, 2))) for _ in range(n)])
    tri = _tri(kitti_cams)
    with _fe(kitti_cams, chunk_frames=3) as off, _fe(kitti_cams, chunk_frames=3, lr_max_diff=1) as fe:
        res, base = fe.stereo_frames(Ls, Rs, Ms), off.stereo_frames(Ls, Rs, Ms)
        for f in range(n):
            assert_checked(res.frame(f), base.frame(f), Ls[f], tri, 1, f"masked frame {f}", fe_off=off if f in (2, 6) else None)
        want = lr.add_new_landmarks(Ls[6], Rs[6], tri, mask=Ms[6], lr_max_diff=1)
        for k in LIVE + ("status",):
            np.testing.assert_array_equal(res.frame(6)[k], want[k], err_msg=k)
        dev = torch.device("cuda:0")
        dL, dR, dM = (torch.from_numpy(a).to(dev) for a in (Ls, Rs, Ms))
        t = dict(n_kp=torch.zeros(n, dtype=torch.int32, device=dev), n_det=torch.zeros(n, dtype=torch.int32, device=dev),
                 uv_l=torch.zeros(n, cap, 2, device=dev), uv_r=torch.zeros(n, cap, 2, device=dev),
                 xyz=torch.zeros(n, cap, 3, dtype=torch.float64, device=dev),
                 dl=torch.zeros(n, cap, 32, dtype=torch.uint8, device=dev), dr=torch.zeros(n, cap, 32, dtype=torch.uint8, device=dev),
                 dist=torch.zeros(n, cap, dtype=torch.int32, device=dev), idx=torch.zeros(n, cap, dtype=torch.int32, device=dev),
                 st=torch.zeros(n, cap, dtype=torch.uint8, device=dev))
        r = _lib.StereoResult(cap, *(t[k].data_ptr() for k in ("n_kp", "n_det", "uv_l", "uv_r", "xyz", "dl", "dr", "dist", "idx", "st")))
        fe.stereo_frames_device(dL.data_ptr(), dR.data_ptr(), W, W * H, n, r, masks_ptr=dM.data_ptr(),
                                stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(t["n_kp"].cpu().numpy(), res.n_keypoints)
        for f in range(n):
            k = int(res.n_keypoints[f])
            for name, key in (("uv_l", "uv_l"), ("dl", "desc_l"), ("dist", "dist"), ("idx", "idx"), ("st", "status")):
                np.testing.assert_array_equal(t[name][f, :k].cpu().numpy(), res.frame(f)[key], err_msg=f"device {f} {key}")
            ok = res.frame(f)["status"] == o.ST_OK
            for name, key in (("uv_r", "uv_r"), ("xyz", "xyz"), ("dr", "desc_r")):
                np.testing.assert_array_equal(t[name][f, :k].cpu().numpy()[ok], res.frame(f)[key][ok], err_msg=f"device {f} {key}")
    Wv, Hv = vi_cams[0].width, vi_cams[0].height
    L, R = stereo_pair(Wv, Hv, 43)
    centres = np.random.default_rng(2).uniform([0, 0], [Wv, Hv], (60, 2)).astype(F32)
    triv = _tri(vi_cams)
    want = lr.add_new_landmarks(L, R, triv, mask=o.mask_active_landmarks(Wv, Hv, centres), lr_max_diff=1)
    with _fe(vi_cams) as off, _fe(vi_cams, lr_max_diff=1) as fe:
        got, base = fe.add_new_landmarks(L, R, mask_centres=centres), off.add_new_landmarks(L, R, mask_centres=centres)
        n_ok, n_rej = assert_checked(got, base, L, triv, 1, "one pair", fe_off=off)
        assert n_ok > 100 and n_rej > 0
        for k in LIVE + ("status",):
            np.testing.assert_array_equal(got[k], want[k], err_msg=k)


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_c5_long_scan_line(kitti_cams):
    """One 3840 x 1080 pair, 10 k corners, 1000-px scan lines: the reverse search takes several windows.  The composed public
    calls cover every slot; the restatement (17 ms of numpy per 1000-px search) every 16th."""
    W, H = 3840, 1080
    cams = _sized(kitti_cams, W, H)
    L, R = stereo_pair(W, H, 3000, d_max=900)
    kw = dict(max_corners=10000, search_range_px=1000.0, max_candidates=131072, chunk_frames=1)
    tri = _tri(cams, search_range=1000.0, max_corners=10000)
    with _fe(cams, **kw) as off, _fe(cams, lr_max_diff=1, **kw) as fe:
        n_ok, n_rej = assert_checked(fe.stereo_frames(L, R).frame(0), off.stereo_frames(L, R).frame(0), L, tri, 1, "C5",
                                     fe_off=off, search=1000.0, every=16)
        assert n_ok > 5000 and n_rej > 0


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_raw_frames_check_on_the_rectified_plane(vi_cams):
    """With rectification set, the reverse search reads the rectified LEFT plane the detector read (svi_rectify gives it;
    svi_triangulate_left rectifies its raw argument the same way)."""
    from svi_mapper_b200.synth import unrectify
    W, H = vi_cams[0].width, vi_cams[0].height
    pairs = [stereo_pair(W, H, 4300 + i) for i in range(3)]
    RL = np.stack([unrectify(p[0], vi_cams[0]) for p in pairs])
    RR = np.stack([unrectify(p[1], vi_cams[1]) for p in pairs])
    tri = _tri(vi_cams)
    with _fe(vi_cams, chunk_frames=2) as off, _fe(vi_cams, chunk_frames=2, lr_max_diff=1) as fe:
        off.set_rectification(*vi_cams)
        fe.set_rectification(*vi_cams)
        L = fe.rectify(RL, 0)
        res, base = fe.stereo_frames(RL, RR), off.stereo_frames(RL, RR)
        for f in range(3):
            n_ok, _ = assert_checked(res.frame(f), base.frame(f), L[f], tri, 1, f"raw frame {f}")
            assert n_ok > 100
            np.testing.assert_array_equal(composed(off, base.frame(f), RL[f], 1), res.frame(f)["status"], err_msg=f"raw composed {f}")


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_check_then_subpixel(kitti_cams, vi_cams):
    """With subpixel_window = subpixel_search = 5 the refinement runs on the slots the check keeps: batch and one-pair
    calls equal the restatement of both modes."""
    W, H = kitti_cams[0].width, kitti_cams[0].height
    Ls, Rs = _batch(W, H, 3, 7500)
    tri = _tri(kitti_cams)
    with _fe(kitti_cams) as off, _fe(kitti_cams, lr_max_diff=1, subpixel_window=5, subpixel_search=5) as fe:
        res, base = fe.stereo_frames(Ls, Rs), off.stereo_frames(Ls, Rs)
        for f in range(3):
            got, ref = res.frame(f), base.frame(f)
            for k in LIVE:
                np.testing.assert_array_equal(got[k], ref[k], err_msg=k)
            st = lr.lr_check(Ls[f], ref["uv_l"], ref["uv_r"], ref["desc_r"], ref["status"], 1, tri)
            uv_r, xyz, st = sp.subpixel_refine(Ls[f], Rs[f], ref["uv_l"], ref["uv_r"], st, 5, 5, tri)
            np.testing.assert_array_equal(got["status"], st)
            ok = st == o.ST_OK
            assert ok.sum() > 300 and (st == lr.ST_LR_INCONSISTENT).sum() > 0
            np.testing.assert_array_equal(got["uv_r"][ok], uv_r[ok])
            np.testing.assert_array_equal(got["xyz"][ok], xyz[ok])
            np.testing.assert_array_equal(got["desc_r"][ok], ref["desc_r"][ok])
    Wv, Hv = vi_cams[0].width, vi_cams[0].height
    L, R = stereo_pair(Wv, Hv, 44)
    triv = _tri(vi_cams)
    want = lr.add_new_landmarks(L, R, triv, lr_max_diff=1, subpixel=(5, 5))
    with _fe(vi_cams, lr_max_diff=1, subpixel_window=5, subpixel_search=5) as fe:
        got = fe.add_new_landmarks(L, R, mask_centres=np.zeros((0, 2), F32))
    for k in LIVE + ("status",):
        np.testing.assert_array_equal(got[k], want[k], err_msg=k)
    ok = want["status"] == o.ST_OK
    for k in OK_ONLY:
        np.testing.assert_array_equal(got[k][ok], want[k][ok], err_msg=k)


def assert_same_results(got, want):
    """Every output svi_stereo_result defines, byte for byte: the per-frame counts, every field of the slots below
    n_keypoints, and uv_right / xyz_left / desc_right of the SVI_OK ones."""
    for k in ("n_keypoints", "n_detected", "n_keypoints_right"):
        if getattr(want, k) is not None:
            np.testing.assert_array_equal(getattr(got, k), getattr(want, k), err_msg=k)
    for f in range(len(want.n_keypoints)):
        g, w = got.frame(f), want.frame(f)
        for k in LIVE + ("status",) + (("second",) if "second" in w else ()):
            np.testing.assert_array_equal(g[k], w[k], err_msg=f"frame {f} {k}")
        ok = w["status"] == o.ST_OK
        for k in OK_ONLY:
            np.testing.assert_array_equal(g[k][ok], w[k][ok], err_msg=f"frame {f} {k}")


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_check_off_sparse_frames_and_refusals(kitti_cams):
    """lr_max_diff = -1 set explicitly is the default ctx (outputs, launches, stage names); the 'lr_check' stage is listed
    and has launches only with the check on; sparse frames give the same bytes with the check on; -2 is refused by
    svi_create and by svi_multi_create."""
    from svi_mapper_b200 import MultiFrontend, SviError, _lib
    W, H = kitti_cams[0].width, kitti_cams[0].height
    Ls, Rs = _batch(W, H, 3, 60)
    with _fe(kitti_cams) as dflt, _fe(kitti_cams, lr_max_diff=-1) as minus1, _fe(kitti_cams, lr_max_diff=2) as on:
        assert dflt.params.lr_max_diff == -1
        for call in (lambda fe: fe.stereo_frames(Ls, Rs), lambda fe: fe.stereo_frames(Ls[:1], Rs[:1])):
            assert_same_results(call(minus1), call(dflt))
        a, b = (fe.add_new_landmarks(Ls[0], Rs[0], mask_centres=np.zeros((0, 2), F32)) for fe in (minus1, dflt))
        for k in LIVE + ("status",):
            np.testing.assert_array_equal(a[k], b[k], err_msg=k)
        for k in OK_ONLY:
            np.testing.assert_array_equal(a[k][b["status"] == o.ST_OK], b[k][b["status"] == o.ST_OK], err_msg=k)
        k_default = (dflt.kernels_per_chunk(64), dflt.kernels_per_chunk(1))
        assert (minus1.kernels_per_chunk(64), minus1.kernels_per_chunk(1)) == k_default
        assert (on.kernels_per_chunk(64), on.kernels_per_chunk(1)) == (k_default[0] + 1, k_default[1] + 1)
        for band, mutual in (((1.0, 1.0, 60.0), False), ((1.0, 1.0, 60.0), True), ((1e9, -1e9, 1e9), True)):
            assert_same_results(on.stereo_frames_sparse(Ls, Rs, None, *band, mutual=mutual),
                                dflt.stereo_frames_sparse(Ls, Rs, None, *band, mutual=mutual))
        names = []
        for fe in (dflt, minus1, on):
            fe.set_profiling(2)
            fe.stereo_frames(Ls, Rs)
            names.append(list(fe.stage_timings()))
        assert names[0] == names[1] == ["harris_box", "boxsum_right", "select_corners", "describe_left", "stereo_match", "subpixel"]
        assert names[2] == ["harris_box", "boxsum_right", "select_corners", "describe_left", "stereo_match", "lr_check", "subpixel"]
        st = on.stage_timings()["lr_check"]
        assert st["launches"] >= 1 and st["total_ms"] > 0
    assert _lib.load().svi_status_text(_lib.SVI_LR_INCONSISTENT).decode().startswith("left-right check")
    with pytest.raises(SviError) as e:
        _fe(kitti_cams, lr_max_diff=-2)
    assert e.value.code == _lib.SVI_ERR_INVALID
    with pytest.raises(SviError) as e:
        MultiFrontend(*kitti_cams, devices=[0], lr_max_diff=-2)
    assert e.value.code == _lib.SVI_ERR_INVALID


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_multi_gpu_equals_one_device(kitti_cams):
    """svi_multi_stereo_frames over two devices == one device, with the check on (needs two visible GPUs)."""
    from svi_mapper_b200 import MultiFrontend, _lib
    if _lib.load().svi_device_count() < 2:
        pytest.skip("needs two visible GPUs")
    W, H = kitti_cams[0].width, kitti_cams[0].height
    Ls, Rs = _batch(W, H, 5, 7600)
    with _fe(kitti_cams, lr_max_diff=1) as one, MultiFrontend(*kitti_cams, devices=[0, 1], lr_max_diff=1) as multi:
        assert_same_results(multi.stereo_frames(Ls, Rs), one.stereo_frames(Ls, Rs))


@pytest.mark.gpu
def test_bounds_checked_build_lr_check():
    """The dense batch and the one-pair parity cases once against the -DSVI_BOUNDS_CHECK build, in which every run-time index
    of lr_check_kernel and of the reverse search is asserted and a failed assertion fails the next call."""
    from svi_mapper_b200 import build as bld
    lib = bld.build_checked()
    env = dict(os.environ, SVI_GPU_LIB=str(lib))
    r = subprocess.run([sys.executable, "-m", "pytest", str(pathlib.Path(__file__)), "-x", "-q", "-m", "gpu",
                        "-k", "dense_batch and kitti_00 or ragged_masked"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "2 passed" in r.stdout and "failed" not in r.stdout
