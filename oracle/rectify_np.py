"""numpy restatement of the reference's image rectification (CStereoCamera.h:102-107, CStereoCameraIMU.h:36-51):
cv::initUndistortRectifyMap(K, D, R, P, (W, H), m1type) and cv::remap(raw, out, map1, map2, INTER_LINEAR) on u8 with the
default BORDER_CONSTANT 0.  CPU reference of libsvi_gpu's svi_rectify_map and rectify_kernel (tests/test_rectify.py pins
both this file and the library against cv2 itself).

init_undistort_rectify_map: OpenCV's scalar loop -- per row i the homogeneous ray (i*ir[1] + ir[2], i*ir[4] + ir[5],
i*ir[7] + ir[8]) with ir = inv(P[:3,:3] @ R) and the column step ir[0] / ir[3] / ir[6] ACCUMULATED, the 4-coefficient
distortion, fp64 throughout; fixed point = cvRound(u * 32) (CV_16SC2) or cvRound(float32(u) * 32) (CV_32FC1 maps as
cv::remap / cv::convertMaps convert them).
remap_linear: OpenCV's fixed-point bilinear path -- initInterTab2D weights rint(float32(1-t) * float32(1-t) * 32768), result
(sum + 2^14) >> 15, taps outside the image read 0."""
from __future__ import annotations

import numpy as np

INTER_BITS = 5
INTER_TAB_SIZE = 1 << INTER_BITS
COEF_BITS = 15
COEF_SCALE = 1 << COEF_BITS


def _cv_round(v: np.ndarray) -> np.ndarray:
    """cvRound of OpenCV's x86 build: half to even; NaN or anything outside int32 -> INT_MIN."""
    v = np.asarray(v, np.float64)
    ok = (v >= -2147483648.0) & (v < 2147483648.0)
    return np.where(ok, np.rint(np.where(ok, v, 0.0)), -2147483648.0).astype(np.int64)


def _inv33(a: np.ndarray) -> np.ndarray:
    """Matx33d::inv: cofactors times 1 / determinant."""
    a = a.reshape(9)
    d = a[0] * (a[4] * a[8] - a[7] * a[5]) - a[1] * (a[3] * a[8] - a[6] * a[5]) + a[2] * (a[3] * a[7] - a[6] * a[4])
    if d == 0 or not np.isfinite(d):
        raise ValueError("singular matrix")
    d = 1.0 / d
    return np.array([(a[4] * a[8] - a[5] * a[7]) * d, (a[2] * a[7] - a[1] * a[8]) * d, (a[1] * a[5] - a[2] * a[4]) * d,
                     (a[5] * a[6] - a[3] * a[8]) * d, (a[0] * a[8] - a[2] * a[6]) * d, (a[2] * a[3] - a[0] * a[5]) * d,
                     (a[3] * a[7] - a[4] * a[6]) * d, (a[1] * a[6] - a[0] * a[7]) * d, (a[0] * a[4] - a[1] * a[3]) * d])


def init_undistort_rectify_map(K, D, R, P, size, float_maps: bool = False):
    """(m1 (H, W, 2) int16, m2 (H, W) uint16) as cv2.initUndistortRectifyMap(K, D, R, P, size, CV_16SC2) returns them, or
    with float_maps as cv2.convertMaps(*cv2.initUndistortRectifyMap(..., CV_32FC1), CV_16SC2)."""
    W, H = int(size[0]), int(size[1])
    K = np.asarray(K, np.float64).reshape(3, 3)
    D = np.asarray(D, np.float64).reshape(4)
    R = np.asarray(R, np.float64).reshape(3, 3)
    P = np.asarray(P, np.float64).reshape(3, -1)
    A = np.zeros((3, 3))
    for i in range(3):                                   # Matx product order
        for j in range(3):
            acc = 0.0
            for k in range(3):
                acc += P[i, k] * R[k, j]
            A[i, j] = acc
    if np.linalg.det(K) == 0:
        raise ValueError("singular K")
    ir = _inv33(A)
    fx, fy, u0, v0 = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    k1, k2, p1, p2 = D
    i = np.arange(H, dtype=np.float64)
    _x, _y, _w = i * ir[1] + ir[2], i * ir[4] + ir[5], i * ir[7] + ir[8]
    u = np.empty((H, W))
    v = np.empty((H, W))
    with np.errstate(all="ignore"):
        for j in range(W):                               # the column step accumulates, as OpenCV's scalar loop does
            w = 1.0 / _w
            x, y = _x * w, _y * w
            x2, y2 = x * x, y * y
            r2 = x2 + y2
            _2xy = 2 * x * y
            kr = (1 + ((0.0 * r2 + k2) * r2 + k1) * r2) / (1 + ((0.0 * r2 + 0.0) * r2 + 0.0) * r2)
            xd = x * kr + p1 * _2xy + p2 * (r2 + 2 * x2) + 0.0 * r2 + 0.0 * r2 * r2
            yd = y * kr + p1 * (r2 + 2 * y2) + p2 * _2xy + 0.0 * r2 + 0.0 * r2 * r2
            u[:, j] = fx * xd + u0
            v[:, j] = fy * yd + v0
            _x, _y, _w = _x + ir[0], _y + ir[3], _w + ir[6]
        if float_maps:
            iu = _cv_round(u.astype(np.float32) * np.float32(INTER_TAB_SIZE))
            iv = _cv_round(v.astype(np.float32) * np.float32(INTER_TAB_SIZE))
        else:
            iu, iv = _cv_round(u * INTER_TAB_SIZE), _cv_round(v * INTER_TAB_SIZE)
    m1 = np.stack([np.clip(iu >> INTER_BITS, -32768, 32767), np.clip(iv >> INTER_BITS, -32768, 32767)], -1).astype(np.int16)
    m2 = ((iv & (INTER_TAB_SIZE - 1)) * INTER_TAB_SIZE + (iu & (INTER_TAB_SIZE - 1))).astype(np.uint16)
    return m1, m2


def inter_tab_2d() -> np.ndarray:
    """initInterTab2D(INTER_LINEAR, fixed point): (32, 32, 4) int64 weights [ty][tx] of the taps (y, x), (y, x+1),
    (y+1, x), (y+1, x+1), with OpenCV's fix-up of a sum that misses 32768 (never needed with 5-bit fractions)."""
    tab = np.zeros((INTER_TAB_SIZE, INTER_TAB_SIZE, 4), np.int64)
    one = np.float32(1)
    for i in range(INTER_TAB_SIZE):
        for j in range(INTER_TAB_SIZE):
            ty, tx = np.float32(i) * (one / np.float32(INTER_TAB_SIZE)), np.float32(j) * (one / np.float32(INTER_TAB_SIZE))
            wy, wx = (one - ty, ty), (one - tx, tx)
            v = np.array([wy[0] * wx[0], wy[0] * wx[1], wy[1] * wx[0], wy[1] * wx[1]], np.float32)
            it = np.rint(v.astype(np.float64) * COEF_SCALE).astype(np.int64)
            diff = int(it.sum()) - COEF_SCALE
            if diff:
                k = int(np.argmax(it)) if diff < 0 else int(np.argmin(it))
                it[k] -= diff
            tab[i, j] = it
    return tab


_TAB = None


def remap_linear(img: np.ndarray, m1: np.ndarray, m2: np.ndarray) -> np.ndarray:
    """cv2.remap(img, m1, m2, INTER_LINEAR) for a u8 (H, W) image and CV_16SC2 maps, BORDER_CONSTANT 0."""
    global _TAB
    if _TAB is None:
        _TAB = inter_tab_2d()
    H, W = img.shape
    sx, sy = m1[..., 0].astype(np.int64), m1[..., 1].astype(np.int64)
    fr = m2.astype(np.int64)
    w = _TAB[(fr >> INTER_BITS) & (INTER_TAB_SIZE - 1), fr & (INTER_TAB_SIZE - 1)]

    def tap(y, x):
        ok = (x >= 0) & (x < W) & (y >= 0) & (y < H)
        return np.where(ok, img[np.clip(y, 0, H - 1), np.clip(x, 0, W - 1)].astype(np.int64), 0)

    acc = tap(sy, sx) * w[..., 0] + tap(sy, sx + 1) * w[..., 1] + tap(sy + 1, sx) * w[..., 2] + tap(sy + 1, sx + 1) * w[..., 3]
    return np.clip((acc + (1 << (COEF_BITS - 1))) >> COEF_BITS, 0, 255).astype(np.uint8)
