"""Image sizes at the edges of the kernels' tiles and runtime parameters other than the reference defaults.

The kernels are built from fixed tiles (Harris 64x32 tiles 62x30 apart, box sums 64x32, bins 128x24, TMA windows 49x120,
passes of 62 candidates, 4 pixels per rectify thread, 16 bytes per mask thread) and each has its own edge code; the
other parity tests run at five image sizes and the default parameters.  Here:

CPU tier: the oracles (numpy and C) against live cv2 at every size of the sweep -- cornerHarris bit for bit (including
calcHarris's scalar tail on the last (W*H) % 4 pixels), goodFeaturesToTrack at several (quality, minDistance, k), FAST.
GPU tier: every image entry point at every size of the sweep against the C oracle (or cv2 / the numpy restatement where
noted), sizes outside [64, 65535] refused, then one runtime parameter at a time at 752x480 and 1243x391."""
import os
import pathlib
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import c_oracle as co
from oracle import frontend_np as o
from svi_mapper_b200.synth import stereo_pair

ROOT = pathlib.Path(__file__).resolve().parents[1]
CALIB = ROOT / "tests" / "golden" / "calib"
F32 = np.float32

# every size with the boundary it sits on (Harris stride 62 x 30, bins 128 x 24, svi_create's range [64, 65535])
SWEEP = [(64, 64), (65, 65),                      # the minimum and one past it
         (124, 90), (1240, 390),                  # exact multiples of the Harris stride
         (125, 91), (126, 92), (127, 93),         # residues 1, 2, 3 past it in both directions
         (185, 89),                               # one short of it
         (256, 96), (257, 97),                    # exact multiple of the bin size, and one past
         (1241, 377),                             # odd height at KITTI width
         (1243, 391),                             # W % 4 == 3
         (4001, 64), (64, 2001)]                  # wide and short, tall and narrow
REFUSED = [(63, 64), (64, 63), (124, 60), (125, 61), (126, 62), (127, 63), (65536, 64), (64, 65536)]   # below / above the range
LIMITS = [(65535, 64), (64, 65535)]
SMALL = [(64, 64), (65, 65), (127, 93), (257, 97)]
# the CPU tier also pins the oracles at the refused small sizes (the stride residues there have H < 64)
CPU_SIZES = SWEEP + [(124, 60), (125, 61), (126, 62), (127, 63)] + LIMITS
CPU_PARAMS = [(0.01, 7.0, 0.04), (0.05, 0.5, 0.02), (0.001, 1.0, 0.15), (0.3, 7.5, 0.06)]   # (quality, minDistance, k)


def _cams(W, H):
    """The KITTI projection matrices with the principal point moved to the centre of a W x H image."""
    from svi_mapper_b200 import load_camera
    out = []
    for side in ("left", "right"):
        P = np.asarray(load_camera(str(CALIB / f"kitti_00_{side}.txt")).P, np.float64).reshape(3, 4).copy()
        P[0, 2], P[1, 2] = W / 2.0, H / 2.0
        out.append(SimpleNamespace(width=W, height=H, P=P))
    return out


def _ids(sizes):
    return [f"{w}x{h}" for w, h in sizes]


@pytest.fixture(scope="module")
def cv2s():
    """cv2 with its scalar dispatch on one thread: the reference's runtime mode (CTrackerGT.cpp:48-49)."""
    import cv2
    opt, threads = cv2.useOptimized(), cv2.getNumThreads()
    cv2.setUseOptimized(False)
    cv2.setNumThreads(1)
    yield cv2
    cv2.setUseOptimized(opt)
    cv2.setNumThreads(threads)


# ------------------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.usefixtures("built_oracle")
@pytest.mark.parametrize("W,H", CPU_SIZES, ids=_ids(CPU_SIZES))
def test_oracles_equal_cv2_at_sweep_sizes(cv2s, W, H):
    """cornerHarris: the C oracle, the numpy OpenCV-order restatement and the exact-sum restatement all equal cv2 bit for
    bit, for four k.  calcHarris evaluates the (continuous) response as one row of W*H pixels -- 4-lane fp32 vectors
    with (float)k, then a scalar tail with the double k for the last (W*H) % 4 pixels -- so at sizes with W*H % 4 != 0
    the last 1-3 pixels of the last row follow another formula; without it they differ from cv2 in the last bit.
    goodFeaturesToTrack (C and numpy) equals cv2 at four (quality, minDistance, k), FAST-9/16 equals cv2's."""
    big = W * H > 1_000_000
    L, _ = stereo_pair(W, H, 7 + W + H)
    tail = (W * H) % 4
    tail_differs = 0
    for k in (0.04, 0.02, 0.06, 0.15):
        want = cv2s.cornerHarris(L, 7, 3, k).view(np.uint32)
        got_c = co.harris_response(L, k=k)
        np.testing.assert_array_equal(got_c.view(np.uint32), want)
        np.testing.assert_array_equal(o.harris_response(L, k, box=o.box7_exact).view(np.uint32), want)
        if not big:
            np.testing.assert_array_equal(o.harris_response(L, k).view(np.uint32), want)
        if tail:   # the vector formula on the tail pixels (what the oracles computed before) is not what cv2 computes
            xx, xy, yy = o.sobel_products(L)
            a, b, c = (o.box7_exact(p).reshape(-1)[-tail:] for p in (xx, xy, yy))
            vec = (a * c - b * b) - (F32(k) * (a + c)) * (a + c)
            tail_differs += int((vec.view(np.uint32) != want.reshape(-1)[-tail:]).sum())
    if (W, H) in ((125, 61), (1241, 377), (1243, 391)):
        assert tail_differs > 0          # seeds picked so that the tail really changes a bit
    for quality, min_distance, k in (CPU_PARAMS[:1] if big else CPU_PARAMS):
        want = cv2s.goodFeaturesToTrack(L, 1000, quality, min_distance, blockSize=7, useHarrisDetector=True, k=k)
        want = np.zeros((0, 2), np.int32) if want is None else want.reshape(-1, 2).astype(np.int32)
        np.testing.assert_array_equal(co.gftt(L, 1000, quality, min_distance, k=k), want, err_msg=str((quality, min_distance, k)))
        if not big:
            np.testing.assert_array_equal(o.gftt(L, 1000, quality, min_distance, k=k), want, err_msg=str((quality, min_distance, k)))
        if quality == 0.01:
            assert len(want) > 0
    for t, nm in ((10, True), (25, False)):
        det = cv2s.FastFeatureDetector_create(threshold=t, nonmaxSuppression=nm, type=cv2s.FAST_FEATURE_DETECTOR_TYPE_9_16)
        want = np.array([[int(p.pt[0]), int(p.pt[1])] for p in det.detect(L)], np.int32).reshape(-1, 2)
        np.testing.assert_array_equal(o.fast9_16(L, t, nm)[0], want)


# ------------------------------------------------------------------------------------------------------------ GPU tier
def _fe(cams, **kw):
    from svi_mapper_b200 import StereoFrontend
    return StereoFrontend(*cams, **kw)


def _compare_frame(got: dict, ref: dict, what=""):
    """Integer / byte outputs bit-exact; xyz within 1e-5 relative and in fact bit-equal (as test_gpu_parity)."""
    assert len(got["uv_l"]) == len(ref["uv_l"]), what
    for k in ("uv_l", "desc_l", "status", "dist", "idx"):
        np.testing.assert_array_equal(got[k], ref[k], err_msg=f"{what} {k}")
    ok = ref["status"] == 0
    for k in ("uv_r", "desc_r"):
        np.testing.assert_array_equal(got[k][ok], ref[k][ok], err_msg=f"{what} {k}")
    if ok.any():
        rel = np.linalg.norm(got["xyz"][ok] - ref["xyz"][ok], axis=1) / np.linalg.norm(ref["xyz"][ok], axis=1)
        assert rel.max() <= 1e-5, what
        np.testing.assert_array_equal(got["xyz"][ok], ref["xyz"][ok], err_msg=f"{what} xyz")


def _pairs(W, H, n, seed):
    p = [stereo_pair(W, H, seed + i) for i in range(n)]
    return np.stack([a for a, _ in p]), np.stack([b for _, b in p])


def _centres(W, H, n, seed):
    """Landmark centres over the image and up to 10 px beyond every edge, some on x.5."""
    rng = np.random.default_rng(seed)
    c = np.stack([rng.uniform(-10, W + 10, n), rng.uniform(-10, H + 10, n)], 1).astype(F32)
    c[: n // 4] = np.floor(c[: n // 4]) + F32(0.5)
    return c


def _torch_result(n, cap, dev):
    import torch
    from svi_mapper_b200 import _lib
    t = dict(n_kp=torch.zeros(n, dtype=torch.int32, device=dev), n_det=torch.zeros(n, dtype=torch.int32, device=dev),
             uv_l=torch.zeros(n, cap, 2, device=dev), uv_r=torch.zeros(n, cap, 2, device=dev),
             xyz=torch.zeros(n, cap, 3, dtype=torch.float64, device=dev),
             dl=torch.zeros(n, cap, 32, dtype=torch.uint8, device=dev), dr=torch.zeros(n, cap, 32, dtype=torch.uint8, device=dev),
             dist=torch.zeros(n, cap, dtype=torch.int32, device=dev), idx=torch.zeros(n, cap, dtype=torch.int32, device=dev),
             st=torch.zeros(n, cap, dtype=torch.uint8, device=dev))
    r = _lib.StereoResult(cap, *(t[k].data_ptr() for k in ("n_kp", "n_det", "uv_l", "uv_r", "xyz", "dl", "dr", "dist", "idx", "st")))
    return t, r


def _result_frame(a: dict, f: int) -> dict:
    n = int(a["n_kp"][f])
    return dict(uv_l=a["uv_l"][f, :n], uv_r=a["uv_r"][f, :n], xyz=a["xyz"][f, :n], desc_l=a["dl"][f, :n], desc_r=a["dr"][f, :n],
                dist=a["dist"][f, :n], idx=a["idx"][f, :n], status=a["st"][f, :n])


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_sizes_and_parameters_outside_the_range_are_refused():
    """svi_create accepts 64 ... 65535 pixels per side (the key packs y << 16 | x) and a positive minimum disparity: at
    min_disparity_px = 0 a zero-disparity match would pass CTriangulator's test and land at infinite depth."""
    from svi_mapper_b200 import SviError, _lib
    for W, H in REFUSED:
        with pytest.raises(SviError, match=r"image size must be within \[64, 65535\]") as e:
            _fe(_cams(W, H))
        assert e.value.code == _lib.SVI_ERR_INVALID
    for v in (0.0, -1.0, float("nan")):
        with pytest.raises(SviError, match="min_disparity_px must be positive") as e:
            _fe(_cams(752, 480), min_disparity_px=v)
        assert e.value.code == _lib.SVI_ERR_INVALID


def _entry_points(W, H, full: bool, **params):
    """Every image entry point of one size against its checker."""
    import torch
    from svi_mapper_b200 import _lib
    cams = _cams(W, H)
    cfg = co.make_config(*cams)
    n = 3 if full else 1
    Ls, Rs = _pairs(W, H, n, 500 + W + H)
    masks = np.full((n, H, W), 255, np.uint8)
    masks[0] = o.mask_active_landmarks(W, H, _centres(W, H, max(4, W * H // 2000), W))
    ref = co.stereo_frames(cfg, Ls, Rs, masks=masks, n_threads=co.host_threads())
    with _fe(cams, chunk_frames=2, **params) as fe:
        # Harris: the exact-sum oracle and the OpenCV-order C oracle (== cv2, test_oracles_equal_cv2_at_sweep_sizes)
        g = fe.harris_response(Ls[0])
        np.testing.assert_array_equal(g.view(np.uint32), o.harris_response(Ls[0], box=o.box7_exact).view(np.uint32))
        np.testing.assert_array_equal(g.view(np.uint32), co.harris_response(Ls[0]).view(np.uint32))
        # detect with and without a mask
        got = fe.detect(Ls, masks)
        for f in range(n):
            np.testing.assert_array_equal(got[f].astype(np.int32), co.gftt(Ls[f], 1000, mask=masks[f]), err_msg=f"detect {f}")
        np.testing.assert_array_equal(fe.detect(Ls[0])[0].astype(np.int32), co.gftt(Ls[0], 1000))
        # the batch (chunks of 2, n not a multiple of it) and the one-pair small call
        res = fe.stereo_frames(Ls, Rs, masks)
        for f in range(n):
            _compare_frame(res.frame(f), co.frame(ref, f), f"batch {f}")
            assert res.n_detected[f] == ref["n_detected"][f]
        one = fe.stereo_frames(Ls[-1], Rs[-1], masks[-1])
        _compare_frame(one.frame(0), co.frame(ref, n - 1), "one pair")
        if not full:
            return
        # describe: points on the 28-px border, one inside it, on x.5
        rng = np.random.default_rng(W * H)
        pts = np.stack([rng.integers(0, W, 300), rng.integers(0, H, 300)], 1).astype(F32)
        pts[:9] = [[28, 28], [27, 28], [W - 29, H - 29], [W - 28, H - 29], [W - 29, H - 28], [28.4, 30.5], [27.5, 28.5],
                   [W - 28.5, H - 28.5], [W / 2 + 0.5, H / 2 - 0.5]]
        pts = np.clip(pts, 0, [W - 1, H - 1]).astype(F32)
        desc, kept = fe.describe(Ls[1], pts)
        keep_ref, desc_ref = co.brief32(Ls[1], pts)
        np.testing.assert_array_equal(np.nonzero(kept)[0], keep_ref)
        np.testing.assert_array_equal(desc[kept], desc_ref)
        # device-resident entry on torch tensors
        dev = torch.device("cuda", 0)
        t, r = _torch_result(n, fe.max_corners, dev)
        dL, dR, dM = (torch.from_numpy(a).to(dev) for a in (Ls, Rs, masks))
        fe.stereo_frames_device(dL.data_ptr(), dR.data_ptr(), W, W * H, n, r, masks_ptr=dM.data_ptr(),
                                stream=torch.cuda.current_stream().cuda_stream)
        fe.check_overflow()
        a = {k: v.cpu().numpy() for k, v in t.items()}
        for f in range(n):
            _compare_frame(_result_frame(a, f), co.frame(ref, f), f"device {f}")
        # padded pitch through the raw host call, garbage in the padding
        pitch = W + 5
        Lp, Rp = np.full((n, H, pitch), 255, np.uint8), np.zeros((n, H, pitch), np.uint8)
        Lp[:, :, :W], Rp[:, :, :W] = Ls, Rs
        cap = fe.max_corners
        h = dict(n_kp=np.zeros(n, np.int32), n_det=np.zeros(n, np.int32), uv_l=np.zeros((n, cap, 2), F32), uv_r=np.zeros((n, cap, 2), F32),
                 xyz=np.zeros((n, cap, 3)), dl=np.zeros((n, cap, 32), np.uint8), dr=np.zeros((n, cap, 32), np.uint8),
                 dist=np.zeros((n, cap), np.int32), idx=np.zeros((n, cap), np.int32), st=np.zeros((n, cap), np.uint8))
        r = _lib.StereoResult(cap, *(h[k].ctypes.data for k in ("n_kp", "n_det", "uv_l", "uv_r", "xyz", "dl", "dr", "dist", "idx", "st")))
        fe.stereo_frames_raw(Lp[1:].ctypes.data, Rp[1:].ctypes.data, pitch, pitch * H, n - 1, r)
        for f in range(n - 1):
            _compare_frame(_result_frame(h, f), co.frame(ref, f + 1), f"padded {f}")
        # the detection mask stamped on the device == cv2.circle (getMaskActiveLandmarks)
        import cv2
        c = _centres(W, H, max(8, W * H // 1500), W + 1)
        m = np.full((H, W), 255, np.uint8)
        for x, y in c:
            cv2.circle(m, (o.cv_round(x), o.cv_round(y)), 7, 0, -1)
        np.testing.assert_array_equal(fe.mask_active_landmarks(c), m)
    return Ls, Rs, masks


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library", "built_oracle")
@pytest.mark.parametrize("W,H", SWEEP, ids=_ids(SWEEP))
def test_size_sweep_entry_points(W, H):
    """Harris, detect (with / without mask), describe, the batch in chunks of 2 (3 frames), the one-pair call, the
    device-resident call on torch tensors, the padded-pitch host call, the device-built mask, FAST mode and the
    sparse-band frames (with / without the left-right check) at one boundary size."""
    import test_sparse_frames as tsf
    import test_sparse_mutual as tsm
    Ls, Rs, masks = _entry_points(W, H, True)
    cams = _cams(W, H)
    # FAST-9/16 (detector = 1) against the cv2-pinned restatement
    with _fe(cams, detector=1, fast_threshold=20, fast_nonmax=1, max_corners=60000, max_candidates=65536, chunk_frames=2) as fe:
        got = fe.detect(Ls, masks)
        for f in range(len(Ls)):
            ref = o.fast9_16(Ls[f], 20, True)[0]
            np.testing.assert_array_equal(got[f].astype(np.int32), ref[masks[f][ref[:, 1], ref[:, 0]] != 0], err_msg=f"fast {f}")
    # sparse-band frames: the numpy restatement of test_sparse_frames / test_sparse_mutual
    tri = tsf._tri(cams)
    with _fe(cams, chunk_frames=2) as fe:
        for band in ((1.0, 1.0, 60.0), (3.0, 0.0, 1e9)):
            for mutual in (False, True):
                res = fe.stereo_frames_sparse(Ls, Rs, masks, *band, mutual=mutual)
                for f in range(len(Ls)):
                    fn = tsm.sparse_frame_mutual_np if mutual else tsf.sparse_frame_np
                    tsf.assert_same(res.frame(f), fn(Ls[f], Rs[f], tri, band, masks[f]), f"sparse {band} {mutual} {f}")


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library", "built_oracle")
@pytest.mark.parametrize("W,H", LIMITS, ids=_ids(LIMITS))
def test_size_limits(W, H):
    """The largest accepted sizes: Harris, detect, the batch and the one-pair call equal the oracle.  A textured frame of
    4 M pixels has more NMS candidates than the default list holds -- a loud capacity error, never a silent drop -- so the
    context gets a longer list (and with it the global-memory selection variant)."""
    from svi_mapper_b200 import SviError
    with pytest.raises(SviError, match="candidate list overflow"):
        _entry_points(W, H, False)
    _entry_points(W, H, False, max_candidates=131072)


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library", "built_oracle")
@pytest.mark.parametrize("W,H", SMALL, ids=_ids(SMALL))
@pytest.mark.parametrize("split,pre,binned", [("1", "0", "0"), ("2", "0", "0"), ("1", "1", "0"), ("2", "1", "0"), ("1", "1", "2")])
def test_size_sweep_matcher_variants(monkeypatch, W, H, split, pre, binned):
    """Every matcher shape forced through the tuning knobs before the context exists, on a batch large enough for the
    batch path (26 frames, one chunk) and on one pair.  fe.config() does not name the matcher; svi_kernels_per_chunk does
    count the LEFT-descriptor kernel and the bin sort, so it proves that the binned kernels (6) and the per-key-point
    ones (4 or 5) are what ran."""
    monkeypatch.setenv("SVI_MATCH_SPLIT", split)
    monkeypatch.setenv("SVI_MATCH_PRE", pre)
    monkeypatch.setenv("SVI_MATCH_BINNED", binned)
    cams = _cams(W, H)
    n = 26
    base_l, base_r = _pairs(W, H, 4, 900 + W)
    Ls, Rs = base_l[np.arange(n) % 4], base_r[np.arange(n) % 4]
    ref = co.stereo_frames(co.make_config(*cams), base_l, base_r, n_threads=co.host_threads())
    with _fe(cams) as fe:
        assert fe.kernels_per_chunk(n) == (6 if binned == "2" else 5 if pre == "1" else 4)
        got = fe.stereo_frames(Ls, Rs)
        one = fe.stereo_frames(Ls[3], Rs[3])
    for f in range(n):
        _compare_frame(got.frame(f), co.frame(ref, f % 4), f"frame {f}")
    _compare_frame(one.frame(0), co.frame(ref, 3), "one pair")
    if W * H > 20000:
        assert sum(int((co.frame(ref, f)["status"] == 0).sum()) for f in range(4)) > 20


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_default_matcher_choice_by_density(monkeypatch):
    """Without the knobs the library picks the binned matcher by key-point density, (W - 56)(H - 56) floored at 1 in the
    denominator: a 64x64 frame counts as dense (binned), a 752x480 one with 1000 corners does not."""
    for v in ("SVI_MATCH_BINNED", "SVI_MATCH_PRE", "SVI_MATCH_SPLIT"):
        monkeypatch.delenv(v, raising=False)
    with _fe(_cams(64, 64)) as fe:
        assert fe.kernels_per_chunk(26) == 6
    with _fe(_cams(752, 480)) as fe:
        assert fe.kernels_per_chunk(26) == 5


def _vi_moved(W, H):
    """vi_sensor's optics (K, distortion, rectification, P) with the principal points moved to the centre of W x H."""
    from svi_mapper_b200 import load_camera
    from svi_mapper_b200.calib import PinholeCamera
    out = []
    for side in ("left", "right"):
        c = load_camera(str(CALIB / f"vi_sensor_{side}.txt"))
        K, P = c.K.copy(), np.asarray(c.P, np.float64).reshape(3, 4).copy()
        dx, dy = (W - c.width) / 2.0, (H - c.height) / 2.0
        K[0, 2] += dx; K[1, 2] += dy
        P[0, 2] += dx; P[1, 2] += dy
        out.append(PinholeCamera(c.label, W, H, P, K, c.focal_length_m, c.distortion, c.rectification))
    return out


RECT_SIZES = [(64, 64), (65, 65), (127, 93), (1243, 391), (64, 2001)]


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
@pytest.mark.parametrize("W,H", RECT_SIZES, ids=_ids(RECT_SIZES))
def test_size_sweep_rectify(cv2s, W, H):
    """svi_rectify == cv2.remap over cv2.initUndistortRectifyMap on vi_sensor optics moved to the new size, integer and
    float maps, W*H a multiple of 8 and not (65x65: 1, 127x93: 3, 1243x391: 5 pixels past it)."""
    cams = _vi_moved(W, H)
    rng = np.random.default_rng(W + H)
    raw = rng.integers(0, 256, (3, H, W), dtype=np.uint8)
    for float_maps in (False, True):
        with _fe(cams, chunk_frames=2) as fe:
            fe.set_rectification(*cams, float_maps=float_maps)
            for side in (0, 1):
                c = cams[side]
                args = (c.K, c.distortion, c.rectification, c.P, (W, H))
                m1, m2 = (cv2s.convertMaps(*cv2s.initUndistortRectifyMap(*args, cv2s.CV_32FC1), cv2s.CV_16SC2) if float_maps
                          else cv2s.initUndistortRectifyMap(*args, cv2s.CV_16SC2))
                want = np.stack([cv2s.remap(r, m1, m2, cv2s.INTER_LINEAR) for r in raw])
                assert fe.rectify(raw, side).tobytes() == want.tobytes(), (side, float_maps)
                assert fe.rectify(raw[1], side).tobytes() == want[1].tobytes(), (side, float_maps)


def _stage2_window_cells(cam, T, xyz, scaling, cell=7):
    """Grid cells of each landmark's stage-2 window (round(round(sqrt|u - c| / 10 + scaling) * 15) half sizes, clipped to
    the image) -- the window-mode selection defers a window with more than 2048 cells to the frame-size configuration."""
    P = np.asarray(cam.P, np.float64).reshape(3, 4)
    X = (T @ np.c_[xyz, np.ones(len(xyz))].T)
    p = P @ X
    u, v = p[0] / p[2], p[1] / p[2]
    hw = np.round(np.round(np.sqrt(np.abs(u - P[0, 2])) / 10.0 + scaling) * 15.0)
    hh = np.round(np.round(np.sqrt(np.abs(v - P[1, 2])) / 10.0 + scaling) * 15.0)
    w = np.minimum(u + hw, cam.width) - np.maximum(u - hw, 0)
    h = np.minimum(v + hh, cam.height) - np.maximum(v - hh, 0)
    return np.ceil(np.maximum(w, 0) / cell) * np.ceil(np.maximum(h, 0) / cell)


TRACK_SIZES = [(65, 65), (127, 93), (257, 97), (1240, 390), (1243, 391), (4001, 64), (64, 2001)]


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library", "built_oracle")
@pytest.mark.parametrize("W,H", TRACK_SIZES, ids=_ids(TRACK_SIZES))
def test_size_sweep_tracking(W, H):
    """track_landmarks stages 1, 2, 3 alone and together against the C port of trackManual, on the landmarks of a frame
    of the same size with per-landmark key-point sizes other than 7: stage-2 windows and epipolar boxes reach the image
    edge at the small sizes, and motion_scaling 12 makes windows of more than 2048 cells (deferred to the frame-size
    selection configuration)."""
    cams = _cams(W, H)
    cfg = co.make_config(*cams)
    L, R = stereo_pair(W, H, 4000 + W)
    ref0 = co.frame(co.stereo_frames(cfg, L, R), 0)
    ok = np.nonzero(ref0["status"] == 0)[0][:150]
    disp = (ref0["uv_l"][ok, 0] - ref0["uv_r"][ok, 0]).astype(F32)
    sizes = np.array([5.0, 6.5, 7.0, 8.0, 10.0], F32)[np.arange(len(ok)) % 5]
    args = (ref0["xyz"][ok], ref0["desc_l"][ok], ref0["desc_r"][ok], disp, sizes)
    kw = dict(uv_reference_left=ref0["uv_l"][ok], desc_reference_left=ref0["desc_l"][ok], T_left_to_world_at_detection=np.eye(4))
    L1, R1 = np.roll(L, (2, 3), axis=(0, 1)), np.roll(R, (2, 3), axis=(0, 1))
    T = np.eye(4)
    T[:3, 3] = (0.015, 0.01, 0.0)
    seen = np.zeros(6, np.int64)
    runs = ((L, R, np.eye(4), 1.0, 1), (L1, R1, np.eye(4), 1.0, 2), (L1, R1, np.eye(4), 1.0, 3), (L, R, T, 1.5, 4),
            (L1, R1, T, 1.5, 7), (L1, R1, np.eye(4), 12.0, 2))
    with _fe(cams) as fe:
        for a, b, pose, scaling, stages in runs:
            want = co.track_landmarks(cfg, a, b, pose, *args, scaling, stages=stages, n_threads=co.host_threads(), **kw)
            got = fe.track_landmarks(a, b, pose, *args, scaling, stages=stages, **kw)
            np.testing.assert_array_equal(got["stage"], want["stage"], err_msg=f"stages {stages} scaling {scaling}")
            np.testing.assert_array_equal(got["status"], want["status"], err_msg=f"stages {stages} scaling {scaling}")
            hit = want["stage"] > 0
            for k in ("uv_l", "uv_r", "xyz", "desc_l", "desc_r"):
                np.testing.assert_array_equal(got[k][hit], want[k][hit], err_msg=f"stages {stages} scaling {scaling} {k}")
            seen += np.bincount(want["stage"], minlength=6)
    if min(W, H) >= 300:
        assert seen[1] > 20 and seen[3] + seen[4] > 5 and seen[5] > 5, seen
    if (W, H) == (1240, 390):
        assert (_stage2_window_cells(cams[0], np.eye(4), ref0["xyz"][ok], 12.0) > 2048).any()


# ------------------------------------------------------------------------------------------------------ parameter sweep
PARAMS = ([("quality_level", v) for v in (0.001, 0.05, 0.3)] + [("harris_k", v) for v in (0.02, 0.06, 0.15)] +
          [("min_distance", v) for v in (0.0, 0.5, 1.0, 7.5, 20.0, 64.5)] +
          [("keypoint_size", v) for v in (5.0, 6.3, 6.5, 8.0, 10.0)] +
          [("search_range_px", v) for v in (0.0, 0.5, 30.5, 61.0, 61.5, 62.0, 124.0, 125.0)] +
          [("match_cutoff", v) for v in (0.0, 1.0, 30.0, 64.5, 257.0)] + [("min_disparity_px", v) for v in (1.0, 50.0)])
ORACLE_NAME = dict(quality_level="quality_level", harris_k="harris_k", min_distance="min_distance", keypoint_size="keypoint_size",
                   search_range_px="search_range", match_cutoff="match_cutoff", min_disparity_px="min_disparity")


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library", "built_oracle")
@pytest.mark.parametrize("W,H", [(752, 480), (1243, 391)], ids=["752x480", "1243x391"])
@pytest.mark.parametrize("field,value", PARAMS, ids=[f"{f}={v}" for f, v in PARAMS])
def test_parameter_sweep(monkeypatch, W, H, field, value):
    """One runtime field of svi_params at a time against co.make_config with the same value: detect, the one-pair call
    and a 24-frame batch (the batch path), the latter once with the library's own matcher choice and once with the binned
    matcher forced where its geometry (4 * keypoint_size integral, ceil(search_range) + 1 <= 62) allows it."""
    cams = _cams(W, H)
    cfg = co.make_config(*cams, **{ORACLE_NAME[field]: value})
    base_l, base_r = _pairs(W, H, 3, 7700)
    n = 24
    Ls, Rs = base_l[np.arange(n) % 3], base_r[np.arange(n) % 3]
    ref = co.stereo_frames(cfg, base_l, base_r, n_threads=co.host_threads())
    kw = {field: value}
    four = 4.0 * float(np.float32(kw.get("keypoint_size", 7.0)))
    rng_ = float(np.float32(kw.get("search_range_px", 60.0)))
    binned_ok = four == np.floor(four) and rng_ > 0 and np.ceil(rng_) + 1 <= 62
    for forced in ("1", "2"):
        monkeypatch.setenv("SVI_MATCH_BINNED", forced)
        with _fe(cams, **kw) as fe:
            if forced == "2":
                assert fe.kernels_per_chunk(n) == (6 if binned_ok else 5)
            got = fe.stereo_frames(Ls, Rs)
            for f in range(n):
                _compare_frame(got.frame(f), co.frame(ref, f % 3), f"{field}={value} binned={forced} frame {f}")
            if forced == "1":
                _compare_frame(fe.stereo_frames(Ls[1], Rs[1]).frame(0), co.frame(ref, 1), f"{field}={value} one pair")
                det = fe.detect(base_l)
                for f in range(3):
                    want = co.gftt(base_l[f], cfg.max_corners, cfg.quality_level, cfg.min_distance, k=cfg.harris_k)
                    np.testing.assert_array_equal(det[f].astype(np.int32), want, err_msg=f"{field}={value} detect {f}")
    n_ok = sum(int((co.frame(ref, f)["status"] == 0).sum()) for f in range(3))
    n_kp = sum(len(co.frame(ref, f)["status"]) for f in range(3))
    assert n_kp > 0
    if field == "match_cutoff" and value == 0.0:
        assert n_ok == 0                       # !(distance < 0): nothing passes the cut-off
    elif field == "keypoint_size" and value < 7.0:
        assert n_ok == 0                       # ROI border 4 * size < BRIEF's 28 px: no candidate keeps a descriptor
    elif not (field == "search_range_px" and value < 1.0):
        assert n_ok > 0


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library", "built_oracle")
@pytest.mark.parametrize("field,value", [("harris_k", 0.15), ("quality_level", 0.05), ("min_distance", 7.5), ("match_cutoff", 64.5)])
def test_parameter_sweep_tracking(field, value):
    """The tracking cascade under a non-default runtime field (stage 2's window detector uses k, quality and
    minDistance; every stage uses its own cut-offs, triangulation the match cut-off), with per-landmark key-point sizes."""
    W, H = 752, 480
    cams = _cams(W, H)
    cfg = co.make_config(*cams, **{ORACLE_NAME[field]: value})
    L, R = stereo_pair(W, H, 4100)
    ref0 = co.frame(co.stereo_frames(cfg, L, R), 0)
    ok = np.nonzero(ref0["status"] == 0)[0][:300]
    disp = (ref0["uv_l"][ok, 0] - ref0["uv_r"][ok, 0]).astype(F32)
    sizes = np.array([6.0, 7.5, 9.0], F32)[np.arange(len(ok)) % 3]
    args = (ref0["xyz"][ok], ref0["desc_l"][ok], ref0["desc_r"][ok], disp, sizes)
    kw = dict(uv_reference_left=ref0["uv_l"][ok], desc_reference_left=ref0["desc_l"][ok], T_left_to_world_at_detection=np.eye(4))
    L1, R1 = np.roll(L, (1, 2), axis=(0, 1)), np.roll(R, (1, 2), axis=(0, 1))
    T = np.eye(4)
    T[:3, 3] = (0.02, 0.01, 0.03)
    seen = np.zeros(6, np.int64)
    with _fe(cams, **{field: value}) as fe:
        for a, b, pose, scaling in ((L, R, np.eye(4), 1.0), (L1, R1, np.eye(4), 1.0), (L1, R1, T, 2.0)):
            want = co.track_landmarks(cfg, a, b, pose, *args, scaling, n_threads=co.host_threads(), **kw)
            got = fe.track_landmarks(a, b, pose, *args, scaling, **kw)
            np.testing.assert_array_equal(got["stage"], want["stage"])
            np.testing.assert_array_equal(got["status"], want["status"])
            hit = want["stage"] > 0
            for k in ("uv_l", "uv_r", "xyz", "desc_l", "desc_r"):
                np.testing.assert_array_equal(got[k][hit], want[k][hit], err_msg=k)
            seen += np.bincount(want["stage"], minlength=6)
    assert seen[1] > 50 and seen[3] + seen[4] > 10, seen


@pytest.mark.gpu
@pytest.mark.usefixtures("built_library")
def test_bounds_checked_build_shapes_and_params():
    """The GPU tests of this file once more against the -DSVI_BOUNDS_CHECK build (every run-time index asserted)."""
    from svi_mapper_b200 import build as bld
    lib = bld.build_checked()
    env = dict(os.environ, SVI_GPU_LIB=str(lib))
    r = subprocess.run([sys.executable, "-m", "pytest", str(pathlib.Path(__file__)), "-x", "-q", "-m", "gpu", "-k", "not bounds_checked"],
                       env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "failed" not in r.stdout
