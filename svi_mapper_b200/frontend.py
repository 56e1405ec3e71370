"""Python host side of the stereo front-end: thin, typed wrappers over the C-ABI of libsvi_gpu.so.

The method names follow the reference's interface for this path
  CFundamentalMatcher::addNewLandmarks        -> StereoFrontend.add_new_landmarks / stereo_frames
  CFundamentalMatcher::trackManual (stage 1)  -> StereoFrontend.track_landmarks
  CTriangulator::getPointTriangulatedInRIGHT  -> StereoFrontend.get_point_triangulated_in_right
  CTriangulator::getPointTriangulatedInLEFT   -> StereoFrontend.get_point_triangulated_in_left
  CTriangulator::getPointInLEFT               -> StereoFrontend.get_point_in_left
  CSolverStereoPosit::getTransformationWORLDtoLEFT -> StereoFrontend.solve_stereo_posit
  cv::GFTTDetector::detect / BRIEF::compute / BFMatcher::match -> detect / describe / match_hamming
Every call goes to the GPU through ctypes; nothing here computes on the CPU."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib


class SviError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libsvi_gpu error {code}: {message}")
        self.code = code


class NoMatchFound(Exception):
    """CExceptionNoMatchFound (src/exceptions/CExceptionNoMatchFound.h) -- raised by the scalar
    convenience wrappers when the per-item status is not SVI_OK, with the reference's text."""

    def __init__(self, status: int):
        self.status = int(status)
        super().__init__(status_text(status))


def status_text(status: int) -> str:
    return _lib.load().svi_status_text(int(status)).decode()


def default_params() -> _lib.Params:
    p = _lib.Params()
    _lib.load().svi_params_default(C.byref(p))
    return p


def _cam(cam) -> _lib.Camera:
    c = _lib.Camera()
    c.width, c.height = int(cam.width), int(cam.height)
    P = np.asarray(cam.P, np.float64).reshape(12)
    for i in range(12):
        c.P[i] = float(P[i])
    return c


def _ptr(a) -> int:
    return a.ctypes.data if a is not None else None


def rectification(cam, float_maps: bool = False) -> _lib.Rectification:
    """svi_rectification of a calib.PinholeCamera: matIntrinsic, vecDistortionCoefficients, matRectification."""
    r = _lib.Rectification()
    for dst, src, n in ((r.K, cam.K, 9), (r.D, cam.distortion, 4), (r.R, cam.rectification, 9)):
        v = np.asarray(src, np.float64).reshape(n)
        for i in range(n):
            dst[i] = float(v[i])
    r.float_maps = 1 if float_maps else 0
    return r


def rectify_map(cam, float_maps: bool = False):
    """svi_rectify_map: the map of one camera as cv::initUndistortRectifyMap(K, D, R, P, (W, H), CV_16SC2) returns it
    -- (xy (H, W, 2) int16, frac (H, W) uint16); with float_maps, the CV_16SC2 form of the CV_32FC1 maps.  Host only."""
    c, r = _cam(cam), rectification(cam, float_maps)
    xy = np.zeros((int(cam.height), int(cam.width), 2), np.int16)
    frac = np.zeros((int(cam.height), int(cam.width)), np.uint16)
    lib = _lib.load()
    rc = lib.svi_rectify_map(C.byref(c), C.byref(r), _ptr(xy), _ptr(frac))
    if rc != _lib.SVI_SUCCESS:
        raise SviError(rc, lib.svi_last_error(None).decode())
    return xy, frac


@dataclass
class StereoFrames:
    """SoA result of the new-landmark path (svi_stereo_result); arrays are (n_frames, capacity, ...)."""
    n_keypoints: np.ndarray
    n_detected: np.ndarray
    uv_left: np.ndarray
    uv_right: np.ndarray
    xyz_left: np.ndarray
    desc_left: np.ndarray
    desc_right: np.ndarray
    distance: np.ndarray
    match_index: np.ndarray
    status: np.ndarray
    second_distance: np.ndarray | None = None     # sparse frames only (stereo_frames_sparse): (n_frames, capacity)
    n_keypoints_right: np.ndarray | None = None   # sparse frames only: (n_frames,)

    @classmethod
    def empty(cls, n: int, cap: int, sparse: bool = False) -> "StereoFrames":
        return cls(n_keypoints=np.zeros(n, np.int32), n_detected=np.zeros(n, np.int32),
                   uv_left=np.zeros((n, cap, 2), np.float32), uv_right=np.zeros((n, cap, 2), np.float32),
                   xyz_left=np.zeros((n, cap, 3), np.float64), desc_left=np.zeros((n, cap, 32), np.uint8),
                   desc_right=np.zeros((n, cap, 32), np.uint8), distance=np.full((n, cap), -1, np.int32),
                   match_index=np.full((n, cap), -1, np.int32), status=np.zeros((n, cap), np.uint8),
                   second_distance=np.full((n, cap), -1, np.int32) if sparse else None,
                   n_keypoints_right=np.zeros(n, np.int32) if sparse else None)

    def result(self) -> _lib.StereoResult:
        """svi_stereo_result over these (host) arrays."""
        return _lib.StereoResult(self.uv_left.shape[1], _ptr(self.n_keypoints), _ptr(self.n_detected), _ptr(self.uv_left),
                                 _ptr(self.uv_right), _ptr(self.xyz_left), _ptr(self.desc_left), _ptr(self.desc_right),
                                 _ptr(self.distance), _ptr(self.match_index), _ptr(self.status))

    def frame(self, f: int) -> dict:
        n = int(self.n_keypoints[f])
        d = dict(uv_l=self.uv_left[f, :n], uv_r=self.uv_right[f, :n], xyz=self.xyz_left[f, :n],
                 desc_l=self.desc_left[f, :n], desc_r=self.desc_right[f, :n], dist=self.distance[f, :n],
                 idx=self.match_index[f, :n], status=self.status[f, :n])
        if self.second_distance is not None:
            d["second"] = self.second_distance[f, :n]
            d["n_right"] = int(self.n_keypoints_right[f])
        return d


class StereoFrontend:
    """One svi_ctx: the GPU-side replacement of CTriangulator + the image-space half of
    CFundamentalMatcher for one stereo camera on one device."""

    def __init__(self, cam_left, cam_right, device: int = 0, lib_path=None, **overrides):
        self._lib = _lib.load(lib_path)   # lib_path: another build of libsvi_gpu.so (e.g. a different BRIEF pair table)
        self.params = _lib.Params()
        self._lib.svi_params_default(C.byref(self.params))
        for k, v in overrides.items():
            if not hasattr(self.params, k):
                raise TypeError(f"unknown svi_params field {k!r}")
            setattr(self.params, k, v)
        self.width, self.height = int(cam_left.width), int(cam_left.height)
        self.max_corners = int(self.params.max_corners)
        self._ctx = C.c_void_p()
        cl, cr = _cam(cam_left), _cam(cam_right)
        rc = self._lib.svi_create(C.byref(cl), C.byref(cr), C.byref(self.params), int(device), C.byref(self._ctx))
        if rc != _lib.SVI_SUCCESS:
            raise SviError(rc, self._lib.svi_last_error(None).decode())

    # -- life cycle
    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._lib.svi_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int):
        if rc != _lib.SVI_SUCCESS:
            raise SviError(rc, self._lib.svi_last_error(self._ctx).decode())

    @property
    def brief_table(self) -> str:
        """svi_brief_table_info: which pair table this library build carries (the shipped one is a stand-in)."""
        return self._lib.svi_brief_table_info().decode()

    def config(self) -> dict:
        a, b, c = C.c_int32(), C.c_int32(), C.c_int32()
        self._check(self._lib.svi_config(self._ctx, C.byref(a), C.byref(b), C.byref(c)))
        return dict(chunk_frames=a.value, n_lanes=b.value, select_in_smem=bool(c.value))

    def kernels_per_chunk(self, n_frames: int) -> int:
        """svi_kernels_per_chunk: kernels launched per chunk of an n_frames call (launch accounting of bench.py)."""
        n = self._lib.svi_kernels_per_chunk(self._ctx, int(n_frames))
        if n < 0:
            self._check(n)
        return n

    def _images(self, img, name):
        a = np.asarray(img)
        if a.dtype != np.uint8:
            raise TypeError(f"{name}: uint8 image expected")
        if a.ndim == 2:
            a = a[None]
        if a.ndim != 3 or a.shape[1] != self.height or a.shape[2] != self.width:
            raise ValueError(f"{name}: expected (n, {self.height}, {self.width}) uint8, got {a.shape}")
        return np.ascontiguousarray(a)

    # -- raw camera images: undistortion + rectification on the device (CStereoCamera.h:102-107)
    def set_rectification(self, cam_left, cam_right, float_maps: bool = False):
        """svi_set_rectification from the two calib.PinholeCamera (K / distortion / rectification; the new camera matrix is
        the P this front-end was created with).  From now on every image argument of every method is a RAW image;
        masks and coordinates stay in the rectified frame.  float_maps: CV_32FC1 maps instead of CV_16SC2."""
        rl, rr = rectification(cam_left, float_maps), rectification(cam_right, float_maps)
        self._check(self._lib.svi_set_rectification(self._ctx, C.byref(rl), C.byref(rr)))

    def clear_rectification(self):
        """Images are rectified already again (the default)."""
        self._check(self._lib.svi_set_rectification(self._ctx, None, None))

    def rectify(self, images, side: int) -> np.ndarray:
        """svi_rectify: raw images (n, H, W) or (H, W) of camera `side` (0 = LEFT, 1 = RIGHT) -> rectified, same shape."""
        a = np.asarray(images)
        A = self._images(a, "images")
        out = np.empty_like(A)
        self._check(self._lib.svi_rectify(self._ctx, int(side), _ptr(A), self.width, self.width * self.height, A.shape[0], _ptr(out), self.width))
        return out[0] if a.ndim == 2 else out

    # -- CFundamentalMatcher::addNewLandmarks for a batch of independent pairs
    def stereo_frames(self, left, right, masks=None, capacity: int | None = None) -> StereoFrames:
        L, R = self._images(left, "left"), self._images(right, "right")
        if L.shape != R.shape:
            raise ValueError("left/right batch shapes differ")
        M = self._images(masks, "masks") if masks is not None else None
        n, cap = L.shape[0], int(capacity or self.max_corners)
        out = StereoFrames(
            n_keypoints=np.zeros(n, np.int32), n_detected=np.zeros(n, np.int32),
            uv_left=np.zeros((n, cap, 2), np.float32), uv_right=np.zeros((n, cap, 2), np.float32),
            xyz_left=np.zeros((n, cap, 3), np.float64), desc_left=np.zeros((n, cap, 32), np.uint8),
            desc_right=np.zeros((n, cap, 32), np.uint8), distance=np.full((n, cap), -1, np.int32),
            match_index=np.full((n, cap), -1, np.int32), status=np.zeros((n, cap), np.uint8))
        r = _lib.StereoResult(cap, _ptr(out.n_keypoints), _ptr(out.n_detected), _ptr(out.uv_left), _ptr(out.uv_right),
                              _ptr(out.xyz_left), _ptr(out.desc_left), _ptr(out.desc_right), _ptr(out.distance),
                              _ptr(out.match_index), _ptr(out.status))
        self._check(self._lib.svi_stereo_frames(self._ctx, _ptr(L), _ptr(R), self.width, self.width * self.height, n,
                                                _ptr(M), C.byref(r)))
        return out

    def _band(self, band_v, min_disparity, max_disparity, mutual=False) -> _lib.SparseBand:
        return _lib.SparseBand(float(band_v), float(min_disparity),
                               float(self.params.search_range_px if max_disparity is None else max_disparity), int(mutual))

    def stereo_frames_sparse(self, left, right, masks=None, band_v: float = 1.0, min_disparity: float = 1.0,
                             max_disparity: float | None = None, capacity: int | None = None, mutual: bool = False) -> StereoFrames:
        """svi_stereo_frames_sparse: the batch of stereo_frames, but every LEFT key-point is matched against the RIGHT
        key-points (same detector, no mask) with |y_L - y_R| <= band_v and min_disparity <= x_L - x_R <= max_disparity
        (default: search_range_px) instead of by a dense scan line.  match_index indexes the frame's RIGHT key-points;
        the result also carries second_distance (for a ratio test) and n_keypoints_right.

        mutual=True adds the left-right check (cv2.BFMatcher crossCheck): a match whose RIGHT key-point has another LEFT
        key-point as its own first arg-min in the same band gets SVI_SPARSE_NOT_MUTUAL.  Status order per slot:
        SVI_TRI_NO_MATCH, SVI_TRI_DISTANCE (the cut-off), SVI_SPARSE_NOT_MUTUAL, then getPointInLEFT (SVI_TRI_ZERO_DISP or
        SVI_OK).  Only status and the OK-only fields (uv_right, xyz_left, desc_right) differ from mutual=False."""
        L, R = self._images(left, "left"), self._images(right, "right")
        if L.shape != R.shape:
            raise ValueError("left/right batch shapes differ")
        M = self._images(masks, "masks") if masks is not None else None
        n, cap = L.shape[0], int(capacity or self.max_corners)
        out = StereoFrames.empty(n, cap, sparse=True)
        r = out.result()
        sp = _lib.SparseResult(_ptr(out.second_distance), _ptr(out.n_keypoints_right))
        band = self._band(band_v, min_disparity, max_disparity, mutual)
        self._check(self._lib.svi_stereo_frames_sparse(self._ctx, _ptr(L), _ptr(R), self.width, self.width * self.height, n, _ptr(M),
                                                       C.byref(band), C.byref(r), C.byref(sp)))
        return out

    def add_new_landmarks(self, img_left, img_right, mask=None, mask_centres=None) -> dict:
        """One pair; per-key-point arrays in the reference's iteration order.  mask_centres (n, 2): the detection mask
        of getMaskActiveLandmarks is built on the GPU from these landmark centres (svi_stereo_frame_masked)."""
        if mask_centres is None:
            return self.stereo_frames(img_left, img_right, mask).frame(0)
        if mask is not None:
            raise ValueError("give either a mask plane or mask centres")
        L, R = self._images(img_left, "left"), self._images(img_right, "right")
        c = np.ascontiguousarray(np.asarray(mask_centres, np.float32).reshape(-1, 2))
        cap = self.max_corners
        out = StereoFrames(
            n_keypoints=np.zeros(1, np.int32), n_detected=np.zeros(1, np.int32),
            uv_left=np.zeros((1, cap, 2), np.float32), uv_right=np.zeros((1, cap, 2), np.float32),
            xyz_left=np.zeros((1, cap, 3), np.float64), desc_left=np.zeros((1, cap, 32), np.uint8),
            desc_right=np.zeros((1, cap, 32), np.uint8), distance=np.full((1, cap), -1, np.int32),
            match_index=np.full((1, cap), -1, np.int32), status=np.zeros((1, cap), np.uint8))
        r = _lib.StereoResult(cap, _ptr(out.n_keypoints), _ptr(out.n_detected), _ptr(out.uv_left), _ptr(out.uv_right),
                              _ptr(out.xyz_left), _ptr(out.desc_left), _ptr(out.desc_right), _ptr(out.distance),
                              _ptr(out.match_index), _ptr(out.status))
        self._check(self._lib.svi_stereo_frame_masked(self._ctx, _ptr(L), _ptr(R), self.width, _ptr(c) if len(c) else None, len(c), C.byref(r)))
        return out.frame(0)

    def mask_active_landmarks(self, centres) -> np.ndarray:
        """getMaskActiveLandmarks: (H, W) u8 plane, 255 with radius-7 zero discs at the centres (built on the GPU)."""
        c = np.ascontiguousarray(np.asarray(centres, np.float32).reshape(-1, 2))
        m = np.empty((self.height, self.width), np.uint8)
        self._check(self._lib.svi_mask_active_landmarks(self._ctx, _ptr(c) if len(c) else None, len(c), _ptr(m), self.width))
        return m

    def stereo_frames_raw(self, left_ptr, right_ptr, pitch, frame_stride, n_frames, result: _lib.StereoResult, masks_ptr=None):
        """svi_stereo_frames on caller-managed HOST memory given as raw addresses (e.g. pinned torch tensors)."""
        self._check(self._lib.svi_stereo_frames(self._ctx, left_ptr, right_ptr, pitch, frame_stride, n_frames, masks_ptr,
                                                C.byref(result)))

    def stereo_frames_device(self, left_ptr, right_ptr, pitch, frame_stride, n_frames, result: _lib.StereoResult,
                             masks_ptr=None, stream: int = 0):
        """svi_stereo_frames_device: all addresses are DEVICE pointers; enqueues after `stream`, no sync."""
        self._check(self._lib.svi_stereo_frames_device(self._ctx, left_ptr, right_ptr, pitch, frame_stride, n_frames,
                                                       masks_ptr, C.byref(result), stream or None))

    def stereo_frames_sparse_device(self, left_ptr, right_ptr, pitch, frame_stride, n_frames, result: _lib.StereoResult,
                                    sparse: _lib.SparseResult, band_v: float = 1.0, min_disparity: float = 1.0,
                                    max_disparity: float | None = None, masks_ptr=None, stream: int = 0, mutual: bool = False):
        """svi_stereo_frames_sparse_device: all addresses (also those in result / sparse) are DEVICE pointers; enqueues after
        `stream`, no sync; capacity overflows surface in check_overflow().  mutual: the left-right check, with the status
        order of stereo_frames_sparse."""
        band = self._band(band_v, min_disparity, max_disparity, mutual)
        self._check(self._lib.svi_stereo_frames_sparse_device(self._ctx, left_ptr, right_ptr, pitch, frame_stride, n_frames, masks_ptr,
                                                              C.byref(band), C.byref(result), C.byref(sparse), stream or None))

    def check_overflow(self):
        """svi_check_overflow: synchronise and raise SviError(SVI_ERR_CAPACITY) if a frame enqueued through
        stereo_frames_device overflowed a candidate list."""
        self._check(self._lib.svi_check_overflow(self._ctx))

    # -- detector / extractor / matcher pieces
    def harris_response(self, img) -> np.ndarray:
        a = self._images(img, "img")[0]
        out = np.empty((self.height, self.width), np.float32)
        self._check(self._lib.svi_harris_response(self._ctx, _ptr(a), self.width, _ptr(out)))
        return out

    def detect(self, imgs, masks=None) -> list[np.ndarray]:
        """cv::GFTTDetector::detect per frame -> list of (k, 2) float32 corner arrays."""
        A = self._images(imgs, "imgs")
        M = self._images(masks, "masks") if masks is not None else None
        n = A.shape[0]
        xy = np.zeros((n, self.max_corners, 2), np.float32)
        counts = np.zeros(n, np.int32)
        self._check(self._lib.svi_detect(self._ctx, _ptr(A), self.width, self.width * self.height, n, _ptr(M), _ptr(xy), _ptr(counts)))
        return [xy[f, :counts[f]].copy() for f in range(n)]

    def describe(self, img, xy):
        """BRIEF-32 at xy (n, 2) -> (desc (n, 32) u8, kept (n,) bool)."""
        a = self._images(img, "img")[0]
        pts = np.ascontiguousarray(np.asarray(xy, np.float32).reshape(-1, 2))
        n = pts.shape[0]
        desc, kept = np.zeros((n, 32), np.uint8), np.zeros(n, np.uint8)
        self._check(self._lib.svi_describe(self._ctx, _ptr(a), self.width, _ptr(pts), n, _ptr(desc), _ptr(kept)))
        return desc, kept.astype(bool)

    def match_hamming(self, query, train):
        q = np.ascontiguousarray(np.asarray(query, np.uint8).reshape(-1, 32))
        t = np.ascontiguousarray(np.asarray(train, np.uint8).reshape(-1, 32))
        idx, dist = np.zeros(len(q), np.int32), np.zeros(len(q), np.int32)
        self._check(self._lib.svi_match_hamming(self._ctx, _ptr(q), len(q), _ptr(t) if len(t) else None, len(t), _ptr(idx), _ptr(dist)))
        return idx, dist

    def match_epipolar(self, query, query_xy, train, train_xy, band_v=1.0, min_disparity=0.0, max_disparity=1e9):
        """Key-point to key-point matching inside an epipolar row band -> (index, distance, second_distance)."""
        q = np.ascontiguousarray(np.asarray(query, np.uint8).reshape(-1, 32))
        t = np.ascontiguousarray(np.asarray(train, np.uint8).reshape(-1, 32))
        qxy = np.ascontiguousarray(np.asarray(query_xy, np.float32).reshape(len(q), 2))
        txy = np.ascontiguousarray(np.asarray(train_xy, np.float32).reshape(len(t), 2))
        idx, dist, second = (np.zeros(len(q), np.int32) for _ in range(3))
        self._check(self._lib.svi_match_epipolar(self._ctx, _ptr(q), _ptr(qxy), len(q), _ptr(t) if len(t) else None,
                                                 _ptr(txy) if len(t) else None, len(t), float(band_v), float(min_disparity),
                                                 float(max_disparity), _ptr(idx), _ptr(dist), _ptr(second)))
        return idx, dist, second

    # -- CTriangulator
    def _tri_out(self, n):
        out = dict(uv=np.zeros((n, 2), np.float32), xyz=np.zeros((n, 3), np.float64), desc=np.zeros((n, 32), np.uint8),
                   dist=np.zeros(n, np.int32), idx=np.zeros(n, np.int32), status=np.zeros(n, np.uint8))
        r = _lib.TriResult(_ptr(out["uv"]), _ptr(out["xyz"]), _ptr(out["desc"]), _ptr(out["dist"]), _ptr(out["idx"]), _ptr(out["status"]))
        return out, r

    def triangulate_right(self, img_right, top_left, uv_left, desc_left, keypoint_size: float = 7.0) -> dict:
        a = self._images(img_right, "img_right")[0]
        tl = np.ascontiguousarray(np.asarray(top_left, np.float32).reshape(-1, 2))
        uv = np.ascontiguousarray(np.asarray(uv_left, np.float32).reshape(-1, 2))
        d = np.ascontiguousarray(np.asarray(desc_left, np.uint8).reshape(-1, 32))
        n = len(tl)
        out, r = self._tri_out(n)
        self._check(self._lib.svi_triangulate_right(self._ctx, _ptr(a), self.width, n, _ptr(tl), _ptr(uv), _ptr(d),
                                                    float(keypoint_size), C.byref(r)))
        return out

    def triangulate_left(self, img_left, search_range, top_left, uv_right, desc_right, keypoint_size: float = 7.0) -> dict:
        a = self._images(img_left, "img_left")[0]
        sr = np.ascontiguousarray(np.asarray(search_range, np.float32).reshape(-1))
        tl = np.ascontiguousarray(np.asarray(top_left, np.float32).reshape(-1, 2))
        uv = np.ascontiguousarray(np.asarray(uv_right, np.float32).reshape(-1, 2))
        d = np.ascontiguousarray(np.asarray(desc_right, np.uint8).reshape(-1, 32))
        n = len(tl)
        out, r = self._tri_out(n)
        self._check(self._lib.svi_triangulate_left(self._ctx, _ptr(a), self.width, n, _ptr(sr), _ptr(tl), _ptr(uv), _ptr(d),
                                                   float(keypoint_size), C.byref(r)))
        return out

    def get_point_triangulated_in_right(self, img_right, u_top_left, v_top_left, keypoint_size, uv_left, desc_left):
        """Scalar form with the reference's argument order (CTriangulator.h:68-73); raises NoMatchFound."""
        r = self.triangulate_right(img_right, [[u_top_left, v_top_left]], [uv_left], [desc_left], keypoint_size)
        if r["status"][0] != _lib.SVI_OK:
            raise NoMatchFound(r["status"][0])
        return r["xyz"][0], r["uv"][0], r["desc"][0]

    def get_point_triangulated_in_left(self, img_left, search_range, u_top_left, v_top_left, keypoint_size, uv_right, desc_right):
        r = self.triangulate_left(img_left, [search_range], [[u_top_left, v_top_left]], [uv_right], [desc_right], keypoint_size)
        if r["status"][0] != _lib.SVI_OK:
            raise NoMatchFound(r["status"][0])
        return r["xyz"][0], r["uv"][0], r["desc"][0]

    def point_in_left(self, uv_left, uv_right):
        a = np.ascontiguousarray(np.asarray(uv_left, np.float32).reshape(-1, 2))
        b = np.ascontiguousarray(np.asarray(uv_right, np.float32).reshape(-1, 2))
        n = len(a)
        xyz, st = np.zeros((n, 3), np.float64), np.zeros(n, np.uint8)
        self._check(self._lib.svi_point_in_left(self._ctx, n, _ptr(a), _ptr(b), _ptr(xyz), _ptr(st)))
        return xyz, st

    def get_point_in_left(self, uv_left, uv_right):
        xyz, st = self.point_in_left([uv_left], [uv_right])
        if st[0] != _lib.SVI_OK:
            raise NoMatchFound(st[0])
        return xyz[0]

    # -- CFundamentalMatcher::trackManual, stage 1
    def track_landmarks(self, img_left, img_right, T_world_to_left, xyz_world, last_desc_left, last_desc_right,
                        last_disparity, keypoint_size, motion_scaling: float, uv_reference_left=None,
                        desc_reference_left=None, T_left_to_world_at_detection=None, stages=None) -> dict:
        """trackManual cascade; stage 3 runs only when the three reference arrays are given.
        stages (bit 0 = stage 1, bit 1 = stage 2, bit 2 = stage 3) restricts the cascade: 3 = the image part of
        getPoseStereoPosit, 4 / 2 = the two branches of trackEpipolar (svi_track_landmarks_stages)."""
        a = self._images(img_left, "img_left")[0]
        b = self._images(img_right, "img_right")[0]
        T = np.ascontiguousarray(np.asarray(T_world_to_left, np.float64).reshape(4, 4))
        xw = np.ascontiguousarray(np.asarray(xyz_world, np.float64).reshape(-1, 3))
        n = len(xw)
        dl = np.ascontiguousarray(np.asarray(last_desc_left, np.uint8).reshape(n, 32))
        dr = np.ascontiguousarray(np.asarray(last_desc_right, np.uint8).reshape(n, 32))
        disp = np.ascontiguousarray(np.asarray(last_disparity, np.float32).reshape(n))
        size = np.ascontiguousarray(np.broadcast_to(np.asarray(keypoint_size, np.float32), (n,)).copy())
        out = dict(status=np.zeros(n, np.uint8), stage=np.zeros(n, np.uint8), uv_l=np.zeros((n, 2), np.float32),
                   uv_r=np.zeros((n, 2), np.float32), xyz=np.zeros((n, 3), np.float64),
                   desc_l=np.zeros((n, 32), np.uint8), desc_r=np.zeros((n, 32), np.uint8))
        uvref = dref = tdet = None
        if uv_reference_left is not None:
            uvref = np.ascontiguousarray(np.asarray(uv_reference_left, np.float64).reshape(n, 2))
            dref = np.ascontiguousarray(np.asarray(desc_reference_left, np.uint8).reshape(n, 32))
            tdet = np.ascontiguousarray(np.broadcast_to(np.asarray(T_left_to_world_at_detection, np.float64), (n, 4, 4)).copy())
        lm = _lib.Landmarks(_ptr(xw), _ptr(dl), _ptr(dr), _ptr(disp), _ptr(size), _ptr(uvref), _ptr(dref), _ptr(tdet))
        r = _lib.TrackResult(_ptr(out["status"]), _ptr(out["stage"]), _ptr(out["uv_l"]), _ptr(out["uv_r"]), _ptr(out["xyz"]),
                             _ptr(out["desc_l"]), _ptr(out["desc_r"]))
        if stages is None:
            self._check(self._lib.svi_track_landmarks(self._ctx, _ptr(a), _ptr(b), self.width, _ptr(T), C.byref(lm), n,
                                                      float(motion_scaling), C.byref(r)))
        else:
            self._check(self._lib.svi_track_landmarks_stages(self._ctx, _ptr(a), _ptr(b), self.width, _ptr(T), C.byref(lm), n,
                                                             float(motion_scaling), int(stages), C.byref(r)))
        return out

    def optimize_landmarks(self, xyz_world_guess, first, pose_index, uv_left, uv_right, proj_world_to_left, proj_world_to_right) -> dict:
        """svi_optimize_landmarks: CLandmark::optimize for n landmarks in one call.  Measurements of landmark i are the entries
        [first[i], first[i + 1]) of pose_index / uv_left / uv_right; pose_index selects a row of the two (n_poses, 3, 4) tables."""
        xg = np.ascontiguousarray(np.asarray(xyz_world_guess, np.float64).reshape(-1, 3))
        n = len(xg)
        fi = np.ascontiguousarray(np.asarray(first, np.int32).reshape(n + 1))
        m = int(fi[-1]) if n else 0
        pi = np.ascontiguousarray(np.asarray(pose_index, np.int32).reshape(m))
        ul = np.ascontiguousarray(np.asarray(uv_left, np.float32).reshape(m, 2))
        ur = np.ascontiguousarray(np.asarray(uv_right, np.float32).reshape(m, 2))
        pl = np.ascontiguousarray(np.asarray(proj_world_to_left, np.float64).reshape(-1, 12))
        pr = np.ascontiguousarray(np.asarray(proj_world_to_right, np.float64).reshape(-1, 12))
        if len(pl) != len(pr):
            raise ValueError("projection tables differ in length")
        out = dict(xyz=np.zeros((n, 3), np.float64), outcome=np.zeros(n, np.uint8), average_squared_error=np.zeros(n, np.float64),
                   iterations=np.zeros(n, np.int32))
        a = _lib.LandmarkMeasurements(_ptr(xg), _ptr(fi), _ptr(pi), _ptr(ul), _ptr(ur), _ptr(pl), _ptr(pr), len(pl))
        r = _lib.OptimizeResult(_ptr(out["xyz"]), _ptr(out["outcome"]), _ptr(out["average_squared_error"]), _ptr(out["iterations"]))
        self._check(self._lib.svi_optimize_landmarks(self._ctx, C.byref(a), n, C.byref(r)))
        return out

    # reason strings of the outcomes (svi_posit_outcome), as the CPU restatement of the solver names them
    POSIT_REASONS = {_lib.SVI_POSIT_OK: None, _lib.SVI_POSIT_TOO_FEW_POINTS: "insufficient number of points",
                     _lib.SVI_POSIT_INACCURATE: "insufficient accuracy", _lib.SVI_POSIT_HIGH_RISK: "inconsistent with prior",
                     _lib.SVI_POSIT_NOT_CONVERGED: "system did not converge"}

    @staticmethod
    def _track_out(n):
        out = dict(status=np.zeros(n, np.uint8), stage=np.zeros(n, np.uint8), uv_l=np.zeros((n, 2), np.float32),
                   uv_r=np.zeros((n, 2), np.float32), xyz=np.zeros((n, 3), np.float64),
                   desc_l=np.zeros((n, 32), np.uint8), desc_r=np.zeros((n, 32), np.uint8))
        r = _lib.TrackResult(_ptr(out["status"]), _ptr(out["stage"]), _ptr(out["uv_l"]), _ptr(out["uv_r"]), _ptr(out["xyz"]),
                             _ptr(out["desc_l"]), _ptr(out["desc_r"]))
        return out, r

    def _posit_dict(self, res) -> dict:
        return dict(T=np.array(res.T_world_to_left[:], np.float64).reshape(4, 4), outcome=int(res.outcome),
                    reason=self.POSIT_REASONS[int(res.outcome)], iterations=int(res.iterations), inliers=int(res.inliers),
                    average_squared_error=float(res.average_squared_error), risk=float(res.risk))

    # -- CTrackerSV: one frame of the stereo-only tracker in one call
    SV_SOURCES = ("posit", "posit-damped", "prior")

    def track_frame_stereo_only(self, img_left, img_right, xyz_world, last_desc_left, last_desc_right, last_disparity, keypoint_size,
                                uv_reference_left, desc_reference_left, T_left_to_world_at_detection, flags, T_estimate,
                                T_estimate_damped, T_last=None, t_imu=None, motion_scaling: float = 1.0) -> dict:
        """svi_track_frame_stereo_only: the pose stage (stages 1-2 and the pose solve around T_estimate, then around
        T_estimate_damped if that fails) and the epipolar stage (stage 3, or the regional stage 2) of one frame in one call.
        Landmark arrays as in track_landmarks (the three reference arrays are required); flags (n,) uint8: bit 0 = pose candidate
        (bIsOptimal), bit 1 = leaves the active set in trackEpipolar.  T_last defaults to T_estimate, t_imu to zero.
        Returns dict(T (4, 4), source ("posit" | "posit-damped" | "prior"), attempts (list of solve_stereo_posit dicts),
        measurements (problem size of each attempt's solve), route (n,) uint8 (svi_sv_route), pose_stage and epipolar_stage
        (track_landmarks dicts over all n landmarks))."""
        a = self._images(img_left, "img_left")[0]
        b = self._images(img_right, "img_right")[0]
        xw = np.ascontiguousarray(np.asarray(xyz_world, np.float64).reshape(-1, 3))
        n = len(xw)
        dl = np.ascontiguousarray(np.asarray(last_desc_left, np.uint8).reshape(n, 32))
        dr = np.ascontiguousarray(np.asarray(last_desc_right, np.uint8).reshape(n, 32))
        disp = np.ascontiguousarray(np.asarray(last_disparity, np.float32).reshape(n))
        size = np.ascontiguousarray(np.broadcast_to(np.asarray(keypoint_size, np.float32), (n,)).copy())
        uvref = np.ascontiguousarray(np.asarray(uv_reference_left, np.float64).reshape(n, 2))
        dref = np.ascontiguousarray(np.asarray(desc_reference_left, np.uint8).reshape(n, 32))
        tdet = np.ascontiguousarray(np.broadcast_to(np.asarray(T_left_to_world_at_detection, np.float64), (n, 4, 4)).copy())
        fl = np.ascontiguousarray(np.asarray(flags, np.uint8).reshape(n))
        Te = np.asarray(T_estimate, np.float64).reshape(16)
        Td = np.asarray(T_estimate_damped, np.float64).reshape(16)
        Tl = Te if T_last is None else np.asarray(T_last, np.float64).reshape(16)
        ti = np.zeros(3) if t_imu is None else np.asarray(t_imu, np.float64).reshape(3)
        fr = _lib.SvFrame(_lib.Landmarks(_ptr(xw), _ptr(dl), _ptr(dr), _ptr(disp), _ptr(size), _ptr(uvref), _ptr(dref), _ptr(tdet)), _ptr(fl))
        for i in range(16):
            fr.T_estimate[i], fr.T_estimate_damped[i], fr.T_last[i] = float(Te[i]), float(Td[i]), float(Tl[i])
        for i in range(3):
            fr.t_imu[i] = float(ti[i])
        fr.motion_scaling = float(motion_scaling)
        pose, rp = self._track_out(n)
        epi, re = self._track_out(n)
        route = np.zeros(n, np.uint8)
        res = _lib.SvFrameResult(pose_stage=rp, route=_ptr(route), epipolar_stage=re)
        self._check(self._lib.svi_track_frame_stereo_only(self._ctx, _ptr(a), _ptr(b), self.width, C.byref(fr), n, C.byref(res)))
        return dict(T=np.array(res.T_world_to_left[:], np.float64).reshape(4, 4), source=self.SV_SOURCES[int(res.source)],
                    attempts=[self._posit_dict(res.attempt[k]) for k in range(int(res.attempts))],
                    measurements=[int(res.measurements[k]) for k in range(int(res.attempts))], route=route, pose_stage=pose,
                    epipolar_stage=epi)

    def solve_stereo_posit(self, xyz_world, uv_left, uv_right, T_estimate, T_last=None, t_imu=None) -> dict:
        """svi_solve_stereo_posit: CSolverStereoPosit::getTransformationWORLDtoLEFT on the GPU -- the WORLD->LEFT pose from n
        stereo measurements (xyz_world (n, 3) float64, uv_left / uv_right (n, 2) float32) starting at the prior T_estimate (4, 4).
        T_last: the previous frame's pose, whose translation a solution within 1 mm of it keeps (default: T_estimate);
        t_imu: the expected translation for the risk test (default: zero).  Returns dict(T (4, 4): the solution, or T_estimate
        when the solve failed; outcome (svi_posit_outcome); reason (None or the failure); iterations; inliers;
        average_squared_error; risk)."""
        xw = np.ascontiguousarray(np.asarray(xyz_world, np.float64).reshape(-1, 3))
        n = len(xw)
        ul = np.ascontiguousarray(np.asarray(uv_left, np.float32).reshape(n, 2))
        ur = np.ascontiguousarray(np.asarray(uv_right, np.float32).reshape(n, 2))
        Te = np.asarray(T_estimate, np.float64).reshape(16)
        Tl = Te if T_last is None else np.asarray(T_last, np.float64).reshape(16)
        ti = np.zeros(3) if t_imu is None else np.asarray(t_imu, np.float64).reshape(3)
        prob = _lib.PositProblem(n, _ptr(xw) if n else None, _ptr(ul) if n else None, _ptr(ur) if n else None)
        for i in range(16):
            prob.T_estimate[i], prob.T_last[i] = float(Te[i]), float(Tl[i])
        for i in range(3):
            prob.t_imu[i] = float(ti[i])
        res = _lib.PositResult()
        self._check(self._lib.svi_solve_stereo_posit(self._ctx, C.byref(prob), C.byref(res)))
        return self._posit_dict(res)

    # -- profiling
    def set_profiling(self, enable):
        """0 / False: off; 1 / True: stage events with overlapping lanes; 2: one lane, exclusive per-kernel durations."""
        self._check(self._lib.svi_set_profiling(self._ctx, int(enable)))

    def stage_timings(self) -> dict:
        names = (C.c_char_p * 8)()
        ms = (C.c_double * 8)()
        cnt = (C.c_int64 * 8)()
        n = self._lib.svi_stage_timings(self._ctx, names, ms, cnt, 8)
        if n < 0:
            self._check(n)
        return {names[i].decode(): dict(total_ms=ms[i], launches=cnt[i]) for i in range(n)}
