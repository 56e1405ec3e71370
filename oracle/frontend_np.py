"""CPU oracle (numpy [+ cv2 where importable]) for svi_mapper's stereo front-end hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under svi_mapper_b200/ imports this module; only
tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs do.

What it restates (all file:line relative to /root/reference):
  * cv::GFTTDetector::create(1000, 0.01, 7.0, 7, true)        src/core/CFundamentalMatcher.cpp:18
    -> harris_response(), gftt()            (OpenCV imgproc arithmetic, SURVEY.md 8a row 1 / App. A)
  * cv::xfeatures2d::BriefDescriptorExtractor::create(32)       src/core/CTriangulator.cpp:11
    -> brief32()                            (OpenCV-contrib algorithm, SURVEY.md 8a row 2)
  * cv::BFMatcher(NORM_HAMMING)::match                           src/core/CTriangulator.cpp:12,93
    -> match_hamming()
  * CTriangulator::getPointTriangulatedInRIGHT[Full]             src/core/CTriangulator.cpp:51-119,185-253
  * CTriangulator::getPointTriangulatedInLEFT (7 args)           src/core/CTriangulator.cpp:255-324
  * CTriangulator::getPointInLEFT                                src/core/CTriangulator.cpp:326-356
  * CFundamentalMatcher::addNewLandmarks                         src/core/CFundamentalMatcher.cpp:83-193
  * CFundamentalMatcher::getMaskActiveLandmarks                  src/core/CFundamentalMatcher.cpp:2043-2073
  * CFundamentalMatcher::trackManual stages 1, 2, 3              src/core/CFundamentalMatcher.cpp:1404-1538, 1545-1785,
    -> track_stage1(), track_manual(), track_stage3(), track_manual_full()                       1786-1993, 2142-2453
  * getPoseStereoPosit / trackEpipolar (image part)              src/core/CFundamentalMatcher.cpp:338-757, 760-1332
    -> track_stages()                       (subsets of the same cascade)
  * CSolverStereoPosit::getTransformationWORLDtoLEFT             src/optimization/CSolverStereoPosit.cpp:8-170
    -> solve_stereo_posit()
  * CLandmark::optimize / _getOptimizedLandmarkSTEREOUV          src/types/CLandmark.cpp:281-296, 447-581
    -> optimize_landmark()
  * optional modes that the reference does not have: fast9_16() (== cv2.FastFeatureDetector), match_epipolar()

Pinning status (SURVEY.md 8c): the reference ships no tests and no golden vectors.
  detect        : pinned against cv2 4.13 (setUseOptimized(False), 1 thread) -- tests/test_oracle_cv2.py
  Hamming/argmin: pinned against cv2.BFMatcher
  mask stencil  : pinned against cv2.circle
  triangulation : pinned against the closed form of src/runnable/triangulation_sampling.cpp:99-120
  BRIEF         : PARITY UNPINNED -- opencv_contrib's generated_32.i pair table is not in this image;
                  the algorithm is restated from the published BRIEF/OpenCV description and uses the
                  stand-in table svi_mapper_b200/brief_pattern_32.txt.
"""
from __future__ import annotations

import math
import pathlib
from dataclasses import dataclass, field

import numpy as np

F32 = np.float32

# ----------------------------------------------------------------------------- status codes
# One value per reference failure string (SURVEY.md Appendix C).  Must match include/svi_gpu.h.
ST_OK = 0
ST_TRI_RANGE = 1      # "<CTriangulator>(getPointTriangulatedIn...) insufficient search range"
ST_TRI_NO_DESC = 2    # "... could not compute descriptors"
ST_TRI_NO_MATCH = 3   # "... no match found"
ST_TRI_DISTANCE = 4   # "... matching distance"
ST_TRI_ZERO_DISP = 5  # "<CTriangulator>(getPointInLEFT) zero disparity"
ST_TRI_BAD_ROI = 6    # ROI leaves the image: the reference dies with cv::Exception here
ST_TRK_DEPTH = 7      # "invalid depth"
ST_TRK_STAGE1_DIST = 8  # "insufficient matching distance"
ST_TRK_TRI_DESC = 9   # "triangulation descriptor mismatch"
ST_TRK_OUT_OF_FOV = 10  # projection outside m_cFieldOfView -> ++uFailedSubsequentTrackings
ST_TRK_NO_FEATURES = 11  # "no features detected"   (stage 2: GFTT found nothing in the window)
ST_TRK_NO_MATCHES = 12   # "no matches found"       (stage 2: every corner was erased by BRIEF's border filter)
ST_TRK_DESC = 13         # "descriptor mismatch"    (stage 2: best corner >= cut-off)
ST_TRK_RANGE = 14        # "out of tracking range"  (stage 2: v - 28 < 0)
ST_EPI_OUT_OF_SIGHT = 15   # CExceptionEpipolarLine "projection out of sight"            :1814
ST_EPI_VERTICAL = 16       # "vertical out of sight"                                      :1845
ST_EPI_NEG_SLOPE = 17      # "caught bad projection negative slope"                       :1871
ST_EPI_POS_SLOPE = 18      # "caught bad projection positive slope"                       :1900
ST_EPI_ZERO_LEN = 19       # "zero line length"                                           :1939
ST_EPI_POOL_EMPTY = 20     # "could not find a matching descriptor (empty key point pool)" :2351
ST_EPI_NO_MATCHES = 21     # "could not find any matches (empty matches pool)"            :2361
ST_EPI_DIST = 22           # "could not find a matching descriptor"                       :2395
ST_EPI_ORIG_DIST = 23      # "... (ORIGINAL matching distance too big)"                   :2390
ST_EPI_NO_TRANSLATION = 24 # detection pose == current pose: the essential matrix is undefined, stage 3 is skipped (:1804)

PATTERN_FILE = pathlib.Path(__file__).resolve().parents[1] / "svi_mapper_b200" / "brief_pattern_32.txt"


def load_pattern(path=PATTERN_FILE) -> np.ndarray:
    rows = [list(map(int, l.split())) for l in open(path) if l.strip() and not l.startswith("#")]
    pat = np.asarray(rows, dtype=np.int32)
    assert pat.shape == (256, 4) and np.abs(pat).max() <= 24
    return pat


PATTERN = load_pattern()


# ----------------------------------------------------------------------------- camera
@dataclass
class Camera:
    """Subset of CPinholeCamera (src/vision/CPinholeCamera.h:16-64)."""
    width: int
    height: int
    P: np.ndarray  # 3x4 float64 m_matProjection
    label: str = ""


@dataclass
class StereoParams:
    """Constants of the hot path (SURVEY.md Appendix B); defaults == reference."""
    max_corners: int = 1000
    quality_level: float = 0.01
    min_distance: float = 7.0
    block_size: int = 7
    harris_k: float = 0.04
    search_range: float = 60.0          # CTriangulator.h:20
    match_cutoff: float = 100.0         # CTriangulator.cpp:13
    min_disparity: float = 0.01         # CTriangulator.h:21
    cutoff_stage1: float = 25.0         # CFundamentalMatcher.cpp:23
    cutoff_stage2: float = 50.0         # CFundamentalMatcher.cpp:24
    cutoff_stage3: float = 50.0         # CFundamentalMatcher.cpp:25
    cutoff_original: float = 100.0      # CFundamentalMatcher.cpp:26
    epipolar_base_length: float = 15.0  # CFundamentalMatcher.h:92
    block_size_stage2: int = 15         # CFundamentalMatcher.h:95 m_uSearchBlockSizePoseOptimization


def _reflect101(i: np.ndarray, n: int) -> np.ndarray:
    i = np.where(i < 0, -i, i)
    return np.where(i >= n, 2 * n - 2 - i, i)


# ----------------------------------------------------------------------------- Harris
_SCALE = 1.0 / (4.0 * 7.0 * 255.0)  # cornerHarris: 1/((1<<(ksize-1))*blockSize) / 255 for CV_8U
_F1 = F32(_SCALE)
_F0 = F32(2.0 * _SCALE)


def sobel_products(img: np.ndarray):
    """Dx, Dy as cv::Sobel(CV_32F, ksize 3, scale) computes them, then the three products.

    Row filter then column filter, every * and + rounded to fp32 separately (no FMA), in the
    operand order validated against cv2 in SURVEY.md Appendix A.1.
    """
    h, w = img.shape
    p = img.astype(F32)
    xi = _reflect101(np.arange(-1, w + 1), w)
    yi = _reflect101(np.arange(-1, h + 1), h)
    pp = p[yi][:, xi]  # (h+2, w+2) padded, REFLECT_101
    # dx=1,dy=0: row kernel [-1,0,1], column kernel [1,2,1]*s (symmetric column filter)
    r = pp[:, 2:] - pp[:, :-2]                                  # exact in fp32
    dx = (r[:-2] + r[2:]) * _F1 + r[1:-1] * _F0
    # dx=0,dy=1: row kernel [1,2,1]*s (generic sequential row filter), column kernel [-1,0,1]
    q = (pp[:, :-2] * _F1 + pp[:, 1:-1] * _F0) + pp[:, 2:] * _F1
    dy = q[2:] - q[:-2]
    assert dx.dtype == F32 and dy.dtype == F32
    return dx * dx, dx * dy, dy * dy


def box7_opencv_order(c: np.ndarray) -> np.ndarray:
    """cv::boxFilter(cov, 7x7, normalize=false, REFLECT_101) on an fp32 plane, in OpenCV's own
    operation order: RowSum<float,double> (running sum along x) then ColumnSum<double,float>
    (running sum along y), both in fp64, one rounding to fp32 at the end."""
    h, w = c.shape
    xi = _reflect101(np.arange(-3, w + 3), w)
    s = c[:, xi].astype(np.float64)  # (h, w+6)
    hs = np.empty((h, w), np.float64)
    acc = np.zeros(h, np.float64)
    for i in range(7):
        acc = acc + s[:, i]
    hs[:, 0] = acc
    for i in range(w - 1):
        acc = acc + (s[:, i + 7] - s[:, i])
        hs[:, i + 1] = acc
    yi = _reflect101(np.arange(-3, h + 3), h)
    hp = hs[yi]  # (h+6, w)
    out = np.empty((h, w), F32)
    acc = np.zeros(w, np.float64)
    for i in range(6):
        acc = acc + hp[i]
    for y in range(h):
        s0 = acc + hp[y + 6]
        out[y] = s0.astype(F32)
        acc = s0 - hp[y]
    return out


def box7_exact(c: np.ndarray) -> np.ndarray:
    """Order-independent variant: plain fp64 sum of the 49 taps, rounded once.  Equal to
    box7_opencv_order whenever no fp64 rounding happens (the common case)."""
    h, w = c.shape
    xi = _reflect101(np.arange(-3, w + 3), w)
    yi = _reflect101(np.arange(-3, h + 3), h)
    s = c[yi][:, xi].astype(np.float64)
    hsum = np.zeros((h + 6, w), np.float64)
    for i in range(7):
        hsum += s[:, i:i + w]
    out = np.zeros((h, w), np.float64)
    for i in range(7):
        out += hsum[i:i + h]
    return out.astype(F32)


def harris_combine(a: np.ndarray, b: np.ndarray, c: np.ndarray, k: float) -> np.ndarray:
    """calcHarris on the three box-summed planes.  OpenCV runs it over the plane as ONE row of W*H pixels (the planes are
    continuous): 4-lane fp32 vectors with (float)k for all but the last (W*H) % 4 pixels, which its scalar tail computes
    as (float)(a*c - b*b - k*(a+c)*(a+c)) with the double k -- a*c, b*b, their difference and a+c in fp32, the rest in
    fp64.  So those 1-3 pixels at the end of the last row can differ from the vector formula in the last bit."""
    kf = F32(k)
    R = (a * c - b * b) - (kf * (a + c)) * (a + c)
    n = R.size
    if n % 4:
        fa, fb, fc, fr = a.reshape(-1), b.reshape(-1), c.reshape(-1), R.reshape(-1)
        for i in range(n - n % 4, n):
            det = float(fa[i] * fc[i] - fb[i] * fb[i])
            tr = float(fa[i] + fc[i])
            fr[i] = F32(det - float(k) * tr * tr)
    return R


def harris_response(img: np.ndarray, k: float = 0.04, box=box7_opencv_order) -> np.ndarray:
    """cv::cornerHarris(img, blockSize 7, ksize 3, k) with optimisations off, fp32 bit-exact."""
    xx, xy, yy = sobel_products(np.ascontiguousarray(img))
    return harris_combine(box(xx), box(xy), box(yy), k)


def harris_response_roi(img: np.ndarray, roi, k: float = 0.04, box=box7_opencv_order) -> np.ndarray:
    """cv::cornerHarris on the ROI view img(roi) of a larger image, as GFTTDetector::detect(img(roi)) runs
    it (CFundamentalMatcher.cpp:1566): the Sobel filters read the parent image's real pixels outside the
    ROI (no BORDER_ISOLATED), the box filter runs on the freshly allocated product planes and therefore
    reflects at the ROI edge.  roi = (x, y, w, h)."""
    x, y, w, h = roi
    xx, xy, yy = sobel_products(np.ascontiguousarray(img))
    a, b, c = (box(np.ascontiguousarray(p[y:y + h, x:x + w])) for p in (xx, xy, yy))
    return harris_combine(a, b, c, k)   # the response of an ROI is a fresh continuous plane: the tail is the window's


def gftt(img: np.ndarray, max_corners=1000, quality=0.01, min_distance=7.0, mask=None,
         response: np.ndarray | None = None, k: float = 0.04) -> np.ndarray:
    """cv::goodFeaturesToTrack(..., useHarrisDetector=true) -> (n,2) int32 (x,y), in cv2's order.

    M = max over mask; threshold TOZERO at float(double(M)*quality); 3x3 dilate equality;
    1-px image border excluded; sort by response desc, ties by larger linear address;
    greedy accept unless an accepted corner lies at squared distance < minDistance^2.
    """
    R = harris_response(img, k) if response is None else response
    h, w = R.shape
    m = np.ones((h, w), bool) if mask is None else (mask != 0)
    if not m.any():
        return np.zeros((0, 2), np.int32)
    M = float(R[m].max())
    thr = F32(M * quality)
    Rt = np.where(R > thr, R, F32(0))
    pad = np.full((h + 2, w + 2), -np.inf, F32)
    pad[1:-1, 1:-1] = Rt
    D = Rt.copy()
    for dy in range(3):
        for dx in range(3):
            D = np.maximum(D, pad[dy:dy + h, dx:dx + w])
    cand = (Rt != 0) & (Rt == D) & m
    cand[0, :] = cand[-1, :] = False
    cand[:, 0] = cand[:, -1] = False
    ys, xs = np.nonzero(cand)
    vals = Rt[ys, xs]
    addr = ys.astype(np.int64) * w + xs
    order = np.lexsort((-addr, -vals.astype(np.float64)))
    ys, xs = ys[order], xs[order]
    md2 = float(min_distance) * float(min_distance)
    if min_distance < 1:
        pts = np.stack([xs, ys], 1)
        return pts[:max_corners].astype(np.int32) if max_corners > 0 else pts.astype(np.int32)
    cell = int(round(min_distance))
    gw, gh = (w + cell - 1) // cell, (h + cell - 1) // cell
    grid = [[] for _ in range(gw * gh)]
    out = []
    for x, y in zip(xs.tolist(), ys.tolist()):
        cx, cy = x // cell, y // cell
        good = True
        for yy in range(max(0, cy - 1), min(gh - 1, cy + 1) + 1):
            for xx in range(max(0, cx - 1), min(gw - 1, cx + 1) + 1):
                for (px, py) in grid[yy * gw + xx]:
                    if (x - px) * (x - px) + (y - py) * (y - py) < md2:
                        good = False
                        break
                if not good:
                    break
            if not good:
                break
        if good:
            grid[cy * gw + cx].append((x, y))
            out.append((x, y))
            if max_corners > 0 and len(out) == max_corners:
                break
    return np.asarray(out, np.int32).reshape(-1, 2)


def detect_cv2(img, max_corners=1000, quality=0.01, min_distance=7.0, mask=None):
    """The genuine OpenCV detector in the reference's runtime mode (CTrackerGT.cpp:48-49)."""
    import cv2
    cv2.setUseOptimized(False)
    cv2.setNumThreads(1)
    det = cv2.GFTTDetector_create(max_corners, quality, min_distance, 7, True)
    kps = det.detect(img, mask)
    return np.asarray([[int(kp.pt[0]), int(kp.pt[1])] for kp in kps], np.int32).reshape(-1, 2)


# ----------------------------------------------------------------------------- FAST-9/16 (optional detector mode)
_FAST_RING = [(0, 3), (1, 3), (2, 2), (3, 1), (3, 0), (3, -1), (2, -2), (1, -3), (0, -3), (-1, -3), (-2, -2), (-3, -1),
              (-3, 0), (-3, 1), (-2, 2), (-1, 3)]   # (dx, dy) of OpenCV's 16-pixel circle, makeOffsets()


def fast9_16(img: np.ndarray, threshold: int = 10, nonmax: bool = True):
    """cv::FAST(img, kps, threshold, nonmax, TYPE_9_16) restated (OpenCV fast.cpp FAST_t<16> + cornerScore<16>):
    a pixel is a corner if >= 9 contiguous circle pixels are all darker than v - t or all brighter than v + t;
    score = largest t for which that still holds; 3x3 non-max suppression with strict >; 3-px border excluded.
    Returns (xy (n,2) int32 in scan order, score (n,) int32).  NOT a reference code path (the reference detects
    with GFTT/Harris): optional mode, pinned against cv2.FastFeatureDetector in tests/test_oracle.py."""
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    t = min(max(int(threshold), 0), 255)
    v = img.astype(np.int32)
    ys, xs = np.mgrid[3:h - 3, 3:w - 3]
    c = v[3:h - 3, 3:w - 3]
    ring = np.stack([v[3 + dy:h - 3 + dy, 3 + dx:w - 3 + dx] for dx, dy in _FAST_RING], 0)   # (16, H-6, W-6)
    ring25 = np.concatenate([ring, ring[:9]], 0)
    d = c[None] - ring25                                                                      # v - ptr[pixel[k]]
    darker = ring25 < (c - t)[None]
    brighter = ring25 > (c + t)[None]

    def has_run9(m):
        run = np.zeros(m.shape[1:], np.int32)
        best = np.zeros(m.shape[1:], np.int32)
        for k in range(25):
            run = np.where(m[k], run + 1, 0)
            best = np.maximum(best, run)
        return best >= 9
    corner = has_run9(darker) | has_run9(brighter)
    # cornerScore<16>
    a0 = np.full(c.shape, t, np.int32)
    for k in range(0, 16, 2):
        a = np.minimum(np.minimum(d[k + 1], d[k + 2]), d[k + 3])
        go = a > a0
        a = np.minimum.reduce([a, d[k + 4], d[k + 5], d[k + 6], d[k + 7], d[k + 8]])
        upd = np.maximum(np.maximum(a0, np.minimum(a, d[k])), np.minimum(a, d[k + 9]))
        a0 = np.where(go, upd, a0)
    b0 = -a0
    for k in range(0, 16, 2):
        b = np.maximum.reduce([d[k + 1], d[k + 2], d[k + 3], d[k + 4], d[k + 5]])
        go = b < b0
        b = np.maximum.reduce([b, d[k + 6], d[k + 7], d[k + 8]])
        upd = np.minimum(np.minimum(b0, np.maximum(b, d[k])), np.maximum(b, d[k + 9]))
        b0 = np.where(go, upd, b0)
    score_in = (-b0 - 1).astype(np.int32)
    score = np.zeros((h, w), np.int32)
    score[3:h - 3, 3:w - 3] = np.where(corner, score_in.astype(np.uint8).astype(np.int32), 0)   # stored as uchar
    cmask = np.zeros((h, w), bool)
    cmask[3:h - 3, 3:w - 3] = corner
    if nonmax:
        pad = np.zeros((h + 2, w + 2), np.int32)
        pad[1:-1, 1:-1] = score
        keep = cmask.copy()
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                if dy or dx:
                    keep &= score > pad[1 + dy:h + 1 + dy, 1 + dx:w + 1 + dx]
        cmask = keep
    yy, xx = np.nonzero(cmask)
    return np.stack([xx, yy], 1).astype(np.int32), score[yy, xx]


# ----------------------------------------------------------------------------- BRIEF
def integral(img: np.ndarray) -> np.ndarray:
    """cv::integral(img, CV_32S): (h+1, w+1) int32."""
    s = np.zeros((img.shape[0] + 1, img.shape[1] + 1), np.int64)
    s[1:, 1:] = np.cumsum(np.cumsum(img.astype(np.int64), 0), 1)
    return s.astype(np.int32)


def cv_round(v: float) -> int:
    """cvRound: round half to even (lrint)."""
    return int(np.rint(np.float64(v)))


def brief32(img: np.ndarray, pts, pattern: np.ndarray = PATTERN):
    """BriefDescriptorExtractor(32)::compute on `img` (an ROI view is just a numpy slice).

    Returns (kept_indices, desc[k,32] u8).  Key-points whose cvRound'ed position is outside
    [28, w-28) x [28, h-28) are erased (KeyPointsFilter::runByImageBorder, PATCH 48 + KERNEL 9);
    the 9x9 box sums are centred on ((int)(y+0.5)+dy, (int)(x+0.5)+dx); test 8j+i -> byte j bit 7-i.
    """
    h, w = img.shape
    pts = np.asarray(pts, F32).reshape(-1, 2)
    keep, cx, cy = [], [], []
    for i, (x, y) in enumerate(pts):
        rx, ry = cv_round(x), cv_round(y)
        sx, sy = int(float(F32(x)) + 0.5), int(float(F32(y)) + 0.5)   # (int)(pt + 0.5), double arithmetic
        # For x.5 coordinates cvRound (half to even) and the sampling centre can differ by one; at the border the
        # reference then reads one column outside its integral image (undefined).  Defined here: erase the point.
        if 28 <= rx < w - 28 and 28 <= ry < h - 28 and 28 <= sx < w - 28 and 28 <= sy < h - 28:
            keep.append(i)
            cx.append(sx)
            cy.append(sy)
    if not keep:
        return np.zeros(0, np.int64), np.zeros((0, 32), np.uint8)
    S = integral(img).astype(np.int64)
    cx = np.asarray(cx)[:, None]
    cy = np.asarray(cy)[:, None]

    def smoothed(dy, dx):
        y = cy + dy[None, :]
        x = cx + dx[None, :]
        return S[y + 5, x + 5] - S[y + 5, x - 4] - S[y - 4, x + 5] + S[y - 4, x - 4]

    bits = smoothed(pattern[:, 0], pattern[:, 1]) < smoothed(pattern[:, 2], pattern[:, 3])
    desc = np.packbits(bits.astype(np.uint8), axis=1, bitorder="big")
    return np.asarray(keep), desc


def boxsum9(img: np.ndarray) -> np.ndarray:
    """9x9 box sum centred at every pixel (valid where the box is inside the image), uint16."""
    h, w = img.shape
    S = integral(img).astype(np.int64)
    out = np.zeros((h, w), np.uint16)
    out[4:h - 4, 4:w - 4] = (S[9:, 9:] - S[9:, :-9] - S[:-9, 9:] + S[:-9, :-9]).astype(np.uint16)
    return out


# ----------------------------------------------------------------------------- matcher
_POP8 = np.array([bin(i).count("1") for i in range(256)], np.int32)


def hamming(a: np.ndarray, b: np.ndarray):
    return _POP8[np.bitwise_xor(a, b)].sum(axis=-1)


def match_hamming(q: np.ndarray, t: np.ndarray):
    """BFMatcher(NORM_HAMMING).match(q 1x32, t Nx32): first arg-min, distance; (-1, -1) if empty."""
    if len(t) == 0:
        return -1, -1
    d = hamming(q.reshape(1, 32), t)
    i = int(np.argmin(d))  # numpy argmin returns the first minimum
    return i, int(d[i])


def match_epipolar(q_desc, q_xy, t_desc, t_xy, band_v=1.0, min_disp=0.0, max_disp=1e9):
    """cv::BFMatcher(NORM_HAMMING).match(query, train, mask) with the epipolar-band mask
    mask[q, t] = |yq - yt| <= band_v and min_disp <= xq - xt <= max_disp, plus the second-best distance.
    Optional mode (not a reference code path); pinned against cv2 in tests/test_oracle.py."""
    q_desc, t_desc = np.asarray(q_desc, np.uint8).reshape(-1, 32), np.asarray(t_desc, np.uint8).reshape(-1, 32)
    q_xy, t_xy = np.asarray(q_xy, F32).reshape(-1, 2), np.asarray(t_xy, F32).reshape(-1, 2)
    idx = np.full(len(q_desc), -1, np.int32)
    dist = np.full(len(q_desc), -1, np.int32)
    second = np.full(len(q_desc), -1, np.int32)
    for i in range(len(q_desc)):
        if len(t_desc) == 0:
            continue
        d = F32(q_xy[i, 0]) - t_xy[:, 0]
        ok = (np.abs(F32(q_xy[i, 1]) - t_xy[:, 1]) <= F32(band_v)) & (d >= F32(min_disp)) & (d <= F32(max_disp))
        cand = np.nonzero(ok)[0]
        if len(cand) == 0:
            continue
        h = hamming(q_desc[i:i + 1], t_desc[cand])
        j = int(np.argmin(h))
        idx[i], dist[i] = cand[j], h[j]
        if len(cand) > 1:
            second[i] = int(np.partition(h, 1)[1])
    return idx, dist, second


# ----------------------------------------------------------------------------- triangulator
class Triangulator:
    """CTriangulator (src/core/CTriangulator.cpp)."""

    def __init__(self, cam_l: Camera, cam_r: Camera, params: StereoParams | None = None):
        self.cl, self.cr = cam_l, cam_r
        self.p = params or StereoParams()
        self.f = float(cam_l.P[0, 0])           # :14
        self.f_inv = 1.0 / self.f               # :15
        self.pu = float(cam_l.P[0, 2])          # :16
        self.pv = float(cam_l.P[1, 2])          # :17
        self.du_r = float(cam_r.P[0, 3])        # :18
        self.du_r_flipped = -self.du_r          # :19
        self.depth_min = self.du_r_flipped / cam_l.width          # :20
        self.depth_max = self.du_r_flipped / self.p.min_disparity  # :21

    def point_in_left(self, uvl, uvr):
        """getPointInLEFT :326-356 -> (status, xyz)."""
        d = F32(uvl[0]) - F32(uvr[0])
        if float(d) < self.p.min_disparity:
            return ST_TRI_ZERO_DISP, None
        z = self.du_r_flipped / float(d)
        x = self.f_inv * z * (float(F32(uvl[0])) - self.pu)
        y = self.f_inv * z * (float(F32(uvl[1])) - self.pv)
        return ST_OK, np.array([x, y, z], np.float64)

    def _search(self, img, u_tl, v_tl, size, n_pool, first_u, width_f):
        """Shared body of :59-117 / :264-322: ROI, pool, BRIEF, match, cut-off."""
        border = F32(4) * F32(size)
        full_h = F32(8) * F32(size) + F32(1)
        roi_w_f = min(F32(n_pool) + full_h, F32(width_f) - F32(u_tl))
        rx, ry, rw, rh = int(F32(u_tl)), int(F32(v_tl)), int(roi_w_f), int(full_h)  # cv::Rect(float..) truncates
        h, w = img.shape
        if rx < 0 or ry < 0 or rw < 0 or rh < 0 or rx + rw > w or ry + rh > h:
            return ST_TRI_BAD_ROI, None
        pool = [(F32(border + F32(first_u) + F32(i)), border) for i in range(n_pool)]
        keep, desc = brief32(img[ry:ry + rh, rx:rx + rw], pool)
        if len(keep) == 0:
            return ST_TRI_NO_DESC, None
        return ST_OK, (pool, keep, desc)

    def triangulate_right(self, img_r, u_tl, v_tl, size, uvl, desc_l):
        """getPointTriangulatedInRIGHT[Full] :51-119/:185-253 -> dict(status, uv, xyz, desc, dist, idx)."""
        u_tl, v_tl = F32(u_tl), F32(v_tl)
        border = F32(4) * F32(size)
        xl = F32(uvl[0])
        if xl <= u_tl + border:
            return dict(status=ST_TRI_RANGE)
        n = int(math.ceil(float(F32(xl - u_tl) - border)))
        st, res = self._search(img_r, u_tl, v_tl, size, n, 0, self.cr.width)
        if st != ST_OK:
            return dict(status=st)
        pool, keep, desc = res
        idx, dist = match_hamming(np.asarray(desc_l, np.uint8), desc)
        if idx < 0:
            return dict(status=ST_TRI_NO_MATCH)
        if not (F32(self.p.match_cutoff) > F32(dist)):
            return dict(status=ST_TRI_DISTANCE, dist=dist, idx=idx)
        px, py = pool[keep[idx]]
        uvr = (F32(px + u_tl), F32(py + v_tl))
        st, xyz = self.point_in_left((xl, F32(uvl[1])), uvr)
        if st != ST_OK:
            return dict(status=st, dist=dist, idx=idx)
        return dict(status=ST_OK, uv=uvr, xyz=xyz, desc=desc[idx].copy(), dist=dist, idx=idx)

    def triangulate_left(self, img_l, search_range, u_tl, v_tl, size, uvr, desc_r):
        """getPointTriangulatedInLEFT (7 args) :255-324."""
        u_tl, v_tl = F32(u_tl), F32(v_tl)
        if 0 >= F32(search_range):
            return dict(status=ST_TRI_RANGE)
        n = int(math.ceil(float(min(F32(search_range), F32(self.cl.width) - u_tl)))) + 1
        st, res = self._search(img_l, u_tl, v_tl, size, n, 1, self.cl.width)
        if st != ST_OK:
            return dict(status=st)
        pool, keep, desc = res
        idx, dist = match_hamming(np.asarray(desc_r, np.uint8), desc)
        if idx < 0:
            return dict(status=ST_TRI_NO_MATCH)
        if not (F32(self.p.match_cutoff) > F32(dist)):
            return dict(status=ST_TRI_DISTANCE, dist=dist, idx=idx)
        px, py = pool[keep[idx]]
        uvl = (F32(px + u_tl), F32(py + v_tl))
        st, xyz = self.point_in_left(uvl, (F32(uvr[0]), F32(uvr[1])))
        if st != ST_OK:
            return dict(status=st, dist=dist, idx=idx)
        return dict(status=ST_OK, uv=uvl, xyz=xyz, desc=desc[idx].copy(), dist=dist, idx=idx)


# ----------------------------------------------------------------------------- addNewLandmarks
def mask_active_landmarks(width, height, centres) -> np.ndarray:
    """getMaskActiveLandmarks :2043-2073: 255 everywhere, filled radius-7 zero discs (cv::circle
    stencil pinned in SURVEY.md A.6: row widths 1,7,9,11,13,13,13,15,13,13,13,11,9,7,1)."""
    half = [0, 3, 4, 5, 6, 6, 6, 7, 6, 6, 6, 5, 4, 3, 0]
    m = np.full((height, width), 255, np.uint8)
    for (cx, cy) in centres:
        cx, cy = cv_round(cx), cv_round(cy)
        for dy in range(-7, 8):
            y = cy + dy
            if 0 <= y < height:
                hw = half[dy + 7]
                x0, x1 = max(cx - hw, 0), min(cx + hw, width - 1)
                if x0 <= x1:
                    m[y, x0:x1 + 1] = 0
    return m


def add_new_landmarks(img_l, img_r, tri: Triangulator, mask=None, use_cv2=False, size=7.0):
    """addNewLandmarks :83-193 minus landmark bookkeeping.  Returns a dict of per-key-point
    arrays in the reference's iteration order (GFTT order after BRIEF's border filter)."""
    p = tri.p
    if use_cv2:
        kps = detect_cv2(img_l, p.max_corners, p.quality_level, p.min_distance, mask)
    else:
        kps = gftt(img_l, p.max_corners, p.quality_level, p.min_distance, mask, k=p.harris_k)
    keep, desc_l = brief32(img_l, kps.astype(F32))                      # :106
    kps = kps[keep] if len(keep) else kps[:0]
    n = len(kps)
    out = dict(uv_l=kps.astype(F32), desc_l=desc_l,
               uv_r=np.zeros((n, 2), F32), xyz=np.zeros((n, 3), np.float64),
               desc_r=np.zeros((n, 32), np.uint8), dist=np.full(n, -1, np.int32),
               idx=np.full(n, -1, np.int32), status=np.zeros(n, np.uint8))
    for u in range(n):
        x, y = F32(kps[u, 0]), F32(kps[u, 1])
        u_tl = max(F32(0), F32(x - F32(p.search_range)) - F32(4) * F32(size))   # :120
        v_tl = y - F32(4) * F32(size)                                            # :121
        r = tri.triangulate_right(img_r, u_tl, v_tl, size, (x, y), desc_l[u])
        out["status"][u] = r["status"]
        out["dist"][u] = r.get("dist", -1)
        out["idx"][u] = r.get("idx", -1)
        if r["status"] == ST_OK:
            out["uv_r"][u] = r["uv"]
            out["xyz"][u] = r["xyz"]
            out["desc_r"][u] = r["desc"]
    return out


# ----------------------------------------------------------------------------- projection helpers
def round_half_away(v) -> F32:
    v = F32(v)
    return F32(math.floor(float(v) + 0.5)) if v >= 0 else F32(-math.floor(float(-v) + 0.5))


def projection_rounded(P: np.ndarray, xyz) -> tuple:
    """CPinholeCamera::getProjectionRounded CPinholeCamera.h:202-210 (std::round on float)."""
    h = P @ np.array([xyz[0], xyz[1], xyz[2], 1.0])
    return round_half_away(F32(h[0] / h[2])), round_half_away(F32(h[1] / h[2]))


def fov_contains(cam: Camera, uv) -> bool:
    """m_cFieldOfView(28,28,W-56,H-56).contains(Point2f) CPinholeCamera.h:61."""
    return 28 <= uv[0] < cam.width - 28 and 28 <= uv[1] < cam.height - 28


def track_stage1(img_l, img_r, tri: Triangulator, T_w2l: np.ndarray, landmarks, motion_scaling: float):
    """trackManual stage 1 (LEFT then RIGHT) :1404-1538 for a list of landmark dicts with keys
    xyz_w (3,), last_desc_l, last_desc_r (32,), last_disparity (float), size (float).
    Returns per-landmark dicts(status, stage, uv_l, uv_r, xyz, desc_l, desc_r)."""
    p = tri.p
    tri_scale = F32(1.0 + motion_scaling)                                     # :1363
    res = []
    for lm in landmarks:
        xyz_l = (T_w2l @ np.append(np.asarray(lm["xyz_w"], np.float64), 1.0))[:3]   # :1404
        uvl = projection_rounded(tri.cl.P, xyz_l)
        uvr = projection_rounded(tri.cr.P, xyz_l)
        size = F32(lm["size"])
        half = F32(4) * size
        search = tri_scale * F32(lm["last_disparity"])                      # :1413
        if not (fov_contains(tri.cl, uvl) and fov_contains(tri.cr, uvr)):
            res.append(dict(status=ST_TRK_OUT_OF_FOV, stage=0))
            continue
        out = None
        # STAGE 1 LEFT :1419-1476
        roi = (F32(uvl[0] - half), F32(uvl[1] - half))
        keep, d = brief32(img_l[int(roi[1]):int(roi[1]) + int(8 * size + 1), int(roi[0]):int(roi[0]) + int(8 * size + 1)], [(half, half)])
        st = ST_TRK_STAGE1_DIST
        if len(keep) == 1 and p.cutoff_stage1 > hamming(np.asarray(lm["last_desc_l"], np.uint8), d[0]):
            r = tri.triangulate_right(img_r, max(F32(0), F32(roi[0] - search)), roi[1], size,
                                      (F32(roi[0] + half), F32(roi[1] + half)), d[0])
            st = r["status"]
            if st == ST_OK:
                z = r["xyz"][2]
                if tri.depth_min > z or tri.depth_max < z:
                    st = ST_TRK_DEPTH
                elif p.cutoff_stage1 < hamming(np.asarray(lm["last_desc_r"], np.uint8), r["desc"]):
                    st = ST_TRK_TRI_DESC
                else:
                    out = dict(status=ST_OK, stage=1, uv_l=(uvl[0], uvl[1]), uv_r=r["uv"], xyz=r["xyz"],
                               desc_l=d[0].copy(), desc_r=r["desc"])
        if out is None:
            # STAGE 1 RIGHT :1480-1538
            roi = (F32(uvr[0] - half), F32(uvr[1] - half))
            keep, d = brief32(img_r[int(roi[1]):int(roi[1]) + int(8 * size + 1), int(roi[0]):int(roi[0]) + int(8 * size + 1)], [(half, half)])
            st = ST_TRK_STAGE1_DIST
            if len(keep) == 1 and p.cutoff_stage1 > hamming(np.asarray(lm["last_desc_r"], np.uint8), d[0]):
                r = tri.triangulate_left(img_l, search, roi[0], roi[1], size,
                                         (F32(roi[0] + half), F32(roi[1] + half)), d[0])
                st = r["status"]
                if st == ST_OK:
                    z = r["xyz"][2]
                    if tri.depth_min > z or tri.depth_max < z:
                        st = ST_TRK_DEPTH
                    elif p.cutoff_stage1 < hamming(np.asarray(lm["last_desc_l"], np.uint8), r["desc"]):
                        st = ST_TRK_TRI_DESC
                    else:
                        out = dict(status=ST_OK, stage=2, uv_l=r["uv"], uv_r=(uvr[0], uvr[1]), xyz=r["xyz"],
                                   desc_l=r["desc"], desc_r=d[0].copy())
        res.append(out if out is not None else dict(status=st, stage=0))
    return res


# ----------------------------------------------------------------------------- trackManual stage 2
def round_half_away_d(v: float) -> float:
    """std::round(double)."""
    return math.floor(v + 0.5) if v >= 0 else -math.floor(-v + 0.5)


def rect_from_points(p1, p2):
    """cv::Rect(cv::Point2f, cv::Point2f): both corners through saturate_cast<int> (cvRound)."""
    x1, y1, x2, y2 = cv_round(p1[0]), cv_round(p1[1]), cv_round(p2[0]), cv_round(p2[1])
    x, y = min(x1, x2), min(y1, y2)
    return x, y, max(x1, x2) - x, max(y1, y2) - y


def stage2_window(cam: Camera, uv, motion_scaling: float, block: int = 15):
    """Search window of stage 2 (:1548-1558): half sizes round(round(w + scaling) * 15) with
    w = sqrt|u - cx| / 10 (CPinholeCamera.h:220-227), corners clamped to the image, as Point2f."""
    wu = math.sqrt(abs(float(uv[0]) - float(cam.P[0, 2]))) / 10.0
    wv = math.sqrt(abs(float(uv[1]) - float(cam.P[1, 2]))) / 10.0
    hw = round_half_away_d(round_half_away_d(wu + motion_scaling) * block)
    hh = round_half_away_d(round_half_away_d(wv + motion_scaling) * block)
    ul = (F32(max(float(uv[0]) - hw, 0.0)), F32(max(float(uv[1]) - hh, 0.0)))
    lr = (F32(min(float(uv[0]) + hw, float(cam.width))), F32(min(float(uv[1]) + hh, float(cam.height))))
    return ul, lr


def track_stage2_side(img_this, img_other, tri: Triangulator, cam_this: Camera, uv_est, last_desc_this, last_desc_other,
                      search, size, motion_scaling: float, left: bool):
    """One side of stage 2 (LEFT :1545-1665, RIGHT :1669-1785) -> dict(status[, uv_this, uv_other, xyz, desc_this, desc_other])."""
    p = tri.p
    size = F32(size)
    half = F32(4) * size
    ul, lr = stage2_window(cam_this, uv_est, motion_scaling, p.block_size_stage2)
    rx, ry, rw, rh = rect_from_points(ul, lr)
    if rw <= 0 or rh <= 0:
        return dict(status=ST_TRK_NO_FEATURES)
    R = harris_response_roi(img_this, (rx, ry, rw, rh), p.harris_k)
    kps = gftt(None, p.max_corners, p.quality_level, p.min_distance, response=R, k=p.harris_k)     # :1566
    if len(kps) == 0:
        return dict(status=ST_TRK_NO_FEATURES)
    wf, hf = F32(cam_this.width), F32(cam_this.height)
    g_ul = (max(F32(ul[0] - half), F32(0)), max(F32(ul[1] - half), F32(0)))                         # :1572-1575
    g_lr = (min(F32(lr[0] + half), wf), min(F32(lr[1] + half), hf))
    gx, gy, gw, gh = rect_from_points(g_ul, g_lr)
    pts = kps.astype(F32) + half                                                                     # :1579
    keep, desc = brief32(img_this[gy:gy + gh, gx:gx + gw], pts)                                      # :1580
    idx, dist = match_hamming(np.asarray(last_desc_this, np.uint8), desc)                            # :1584
    if idx < 0:
        return dict(status=ST_TRK_NO_MATCHES)
    if not (p.cutoff_stage2 > dist):
        return dict(status=ST_TRK_DESC)
    best = pts[keep[idx]]
    in_cam = (F32(F32(ul[0] + best[0]) - half), F32(F32(ul[1] + best[1]) - half))                    # :1592
    d_this = desc[idx]
    v_ref = F32(in_cam[1] - half)
    if not (0.0 <= v_ref):
        return dict(status=ST_TRK_RANGE)
    if left:
        r = tri.triangulate_right(img_other, max(F32(0), F32(F32(in_cam[0] - F32(search)) - half)), v_ref, size, in_cam, d_this)
    else:
        r = tri.triangulate_left(img_other, search, max(F32(0), F32(in_cam[0] - half)), v_ref, size, in_cam, d_this)
    if r["status"] != ST_OK:
        return dict(status=r["status"])
    z = r["xyz"][2]
    if tri.depth_min > z or tri.depth_max < z:
        return dict(status=ST_TRK_DEPTH)
    if not (p.cutoff_stage2 > hamming(np.asarray(last_desc_other, np.uint8), r["desc"])):
        return dict(status=ST_TRK_TRI_DESC)
    return dict(status=ST_OK, uv_this=in_cam, uv_other=r["uv"], xyz=r["xyz"], desc_this=d_this.copy(), desc_other=r["desc"])


def fov_gate(tri: Triangulator, T_w2l: np.ndarray, landmarks):
    """The gate in front of stages 1 and 2 (:1416, :1036): both rounded projections inside the field of view."""
    res = []
    for lm in landmarks:
        xyz_l = (T_w2l @ np.append(np.asarray(lm["xyz_w"], np.float64), 1.0))[:3]
        ok = fov_contains(tri.cl, projection_rounded(tri.cl.P, xyz_l)) and fov_contains(tri.cr, projection_rounded(tri.cr.P, xyz_l))
        res.append(dict(status=ST_TRK_STAGE1_DIST if ok else ST_TRK_OUT_OF_FOV, stage=0))
    return res


def track_manual(img_l, img_r, tri: Triangulator, T_w2l: np.ndarray, landmarks, motion_scaling: float, stage1: bool = True):
    """trackManual stages 1 and 2 (:1404-1785) as a first-success cascade; stage codes
    1 = stage 1 LEFT, 2 = stage 1 RIGHT, 3 = stage 2 LEFT, 4 = stage 2 RIGHT, 0 = not tracked (stage 3 is the caller's).
    This is also the image part of getPoseStereoPosit (:338-757, the same two stages on the optimal landmarks);
    stage1=False leaves only the gate and stage 2 = the zero-translation branch of trackEpipolar (:1022-1290)."""
    s1 = track_stage1(img_l, img_r, tri, T_w2l, landmarks, motion_scaling) if stage1 else fov_gate(tri, T_w2l, landmarks)
    tri_scale = F32(1.0 + motion_scaling)
    out = []
    for lm, r1 in zip(landmarks, s1):
        if r1["stage"] or r1["status"] == ST_TRK_OUT_OF_FOV:
            out.append(r1)
            continue
        xyz_l = (T_w2l @ np.append(np.asarray(lm["xyz_w"], np.float64), 1.0))[:3]
        uvl, uvr = projection_rounded(tri.cl.P, xyz_l), projection_rounded(tri.cr.P, xyz_l)
        search = tri_scale * F32(lm["last_disparity"])
        r = track_stage2_side(img_l, img_r, tri, tri.cl, uvl, lm["last_desc_l"], lm["last_desc_r"], search, lm["size"], motion_scaling, True)
        if r["status"] == ST_OK:
            out.append(dict(status=ST_OK, stage=3, uv_l=r["uv_this"], uv_r=r["uv_other"], xyz=r["xyz"], desc_l=r["desc_this"], desc_r=r["desc_other"]))
            continue
        r = track_stage2_side(img_r, img_l, tri, tri.cr, uvr, lm["last_desc_r"], lm["last_desc_l"], search, lm["size"], motion_scaling, False)
        if r["status"] == ST_OK:
            out.append(dict(status=ST_OK, stage=4, uv_l=r["uv_other"], uv_r=r["uv_this"], xyz=r["xyz"], desc_l=r["desc_other"], desc_r=r["desc_this"]))
        else:
            out.append(dict(status=r["status"], stage=0))
    return out


# ----------------------------------------------------------------------------- trackManual stage 3
def _mul3(A, B):
    """3x3 product, every element ((a0*b0 + a1*b1) + a2*b2) -- the order the host C++ uses."""
    return [[(A[i][0] * B[0][j] + A[i][1] * B[1][j]) + A[i][2] * B[2][j] for j in range(3)] for i in range(3)]


def _inv3(m):
    """3x3 inverse by cofactors (adjugate / determinant), the closed form Eigen uses for fixed 3x3."""
    def cof(i, j):
        i1, i2, j1, j2 = (i + 1) % 3, (i + 2) % 3, (j + 1) % 3, (j + 2) % 3
        return m[i1][j1] * m[i2][j2] - m[i1][j2] * m[i2][j1]
    c0 = [cof(0, 0), cof(1, 0), cof(2, 0)]
    det = (c0[0] * m[0][0] + c0[1] * m[1][0]) + c0[2] * m[2][0]
    inv_det = 1.0 / det
    return [[cof(j, i) * inv_det for j in range(3)] for i in range(3)]


def _ieee_div(a: float, b: float) -> float:
    """a / b with C semantics (inf / nan instead of ZeroDivisionError)."""
    if b != 0.0:
        return a / b
    if a != a or a == 0.0:
        return float("nan")
    return math.copysign(float("inf"), a) * math.copysign(1.0, b)


def epipolar_plan(tri: Triangulator, T_w2l, T_det_l2w, uv_ref, xyz_w, motion_scaling: float):
    """Geometry of stage 3 up to the sampling request (:1795-1947) in plain double arithmetic.
    Returns dict(status) or dict(status=ST_OK, along_u, start, count, coeff)."""
    p = tri.p
    Tw = [[float(T_w2l[i][j]) for j in range(4)] for i in range(4)]
    Td = [[float(T_det_l2w[i][j]) for j in range(4)] for i in range(4)]
    R = [[(Tw[i][0] * Td[0][j] + Tw[i][1] * Td[1][j]) + Tw[i][2] * Td[2][j] for j in range(3)] for i in range(3)]
    t = [((Tw[i][0] * Td[0][3] + Tw[i][1] * Td[1][3]) + Tw[i][2] * Td[2][3]) + Tw[i][3] for i in range(3)]
    if not (0.0 < (t[0] * t[0] + t[1] * t[1]) + t[2] * t[2]):
        return dict(status=ST_EPI_NO_TRANSLATION)
    S = [[0.0, -t[2], t[1]], [t[2], 0.0, -t[0]], [-t[1], t[0], 0.0]]          # CMiniVisionToolbox::getSkew
    E = _mul3(R, S)                                                           # :1800
    P = tri.cl.P
    K = [[float(P[i, j]) for j in range(3)] for i in range(3)]                # m_matIntrinsicP
    Ki = _inv3(K)
    KiT = [[Ki[j][i] for j in range(3)] for i in range(3)]
    F = _mul3(_mul3(KiT, E), Ki)                                              # :1801
    u0, v0 = float(uv_ref[0]), float(uv_ref[1])
    c = [(F[i][0] * u0 + F[i][1] * v0) + F[i][2] * 1.0 for i in range(3)]      # :1818
    xyz_l = [((Tw[i][0] * float(xyz_w[0]) + Tw[i][1] * float(xyz_w[1])) + Tw[i][2] * float(xyz_w[2])) + Tw[i][3] for i in range(3)]
    proj = projection_rounded(tri.cl.P, xyz_l)                                # :1807
    if not fov_contains(tri.cl, proj):
        return dict(status=ST_EPI_OUT_OF_SIGHT)
    W, H = float(tri.cl.width), float(tri.cl.height)
    half = 10.0 * motion_scaling                                              # :1362
    wu = math.sqrt(abs(float(proj[0]) - float(P[0, 2]))) / 10.0
    wv = math.sqrt(abs(float(proj[1]) - float(P[1, 2]))) / 10.0
    hl_u = p.epipolar_base_length + wu * half                                 # :1821-1822
    hl_v = p.epipolar_base_length + wv * half

    def curve_v(u):
        return _ieee_div(-(c[0] * u + c[2]), c[1])

    def curve_u(v):
        return _ieee_div(-(c[1] * v + c[2]), c[0])

    u_min_raw = max(float(proj[0]) - hl_u, 0.0)
    u_max_raw = min(float(proj[0]) + hl_u, W)
    v_min_raw, v_max_raw = curve_v(u_min_raw), curve_v(u_max_raw)
    if (0.0 > v_min_raw and 0.0 > v_max_raw) or (H < v_min_raw and H < v_max_raw):
        return dict(status=ST_EPI_VERTICAL)
    v_lim_min = max(float(proj[1]) - hl_v, 0.0)
    v_lim_max = min(float(proj[1]) + hl_v, H)
    u_min, u_max = u_min_raw, u_max_raw
    if v_min_raw < v_max_raw:
        if v_lim_min > v_max_raw or v_lim_max < v_min_raw:
            return dict(status=ST_EPI_NEG_SLOPE)
        if v_lim_min > v_min_raw:
            v_for_min = v_lim_min
            u_min = curve_u(v_for_min)
        else:
            v_for_min = v_min_raw
        if v_lim_max < v_max_raw:
            v_for_max = v_lim_max
            u_max = curve_u(v_for_max)
        else:
            v_for_max = v_max_raw
    else:
        if v_lim_min > v_min_raw or v_lim_max < v_max_raw:
            return dict(status=ST_EPI_POS_SLOPE)
        if v_lim_min > v_max_raw:
            v_for_min = v_lim_min
            u_max = curve_u(v_for_min)
        else:
            v_for_min = v_max_raw
        if v_lim_max < v_min_raw:
            v_for_max = v_lim_max
            u_min = curve_u(v_for_max)
        else:
            v_for_max = v_min_raw
    du, dv = u_max - u_min, v_for_max - v_for_min
    if not (math.isfinite(du) and math.isfinite(dv)) or du < 0.0 or dv < 0.0 or du >= 65536.0 or dv >= 65536.0:
        return dict(status=ST_EPI_ZERO_LEN)   # the reference's uint32 conversion is undefined here
    delta_u, delta_v = int(du), int(dv)                                       # uint32_t truncation :1933-1934
    if delta_u == 0 and delta_v == 0:
        return dict(status=ST_EPI_ZERO_LEN)
    if delta_v < delta_u:
        return dict(status=ST_OK, along_u=True, start=u_min, count=delta_u, coeff=c)
    return dict(status=ST_OK, along_u=False, start=v_for_min, count=delta_v, coeff=c)


def epipolar_match(img, tri: Triangulator, plan, size, last_desc, orig_desc):
    """_getMatchSampleRecursiveU/V + _getMatch (:2142-2397): one key-point per pixel along the line, BRIEF in the
    bounding ROI, 1 x N match, cut-offs 50 (last) / 100 (original); one retry with the samples moved by +2 px."""
    p = tri.p
    c = plan["coeff"]
    n = plan["count"]
    size = F32(size)
    wf, hf = F32(tri.cl.width), F32(tri.cl.height)
    h, w = img.shape
    status = ST_EPI_POOL_EMPTY
    for off in (0, 2):                                                        # recursion depth 0, then 2 (limit 2, step 2)
        pool = []
        for i in range(n):
            if plan["along_u"]:
                du = plan["start"] + i
                dv = _ieee_div(-(c[0] * du + c[2]), c[1]) + off
            else:
                dv = plan["start"] + i
                du = _ieee_div(-(c[1] * dv + c[2]), c[0]) + off
            pool.append((F32(du), F32(dv)))
        centre = pool[n // 2]
        f_du = F32(abs(F32(pool[0][0] - pool[-1][0]))) + F32(16) * size
        f_dv = F32(abs(F32(pool[0][1] - pool[-1][1]))) + F32(16) * size
        u_tl = max(F32(centre[0] - f_du / F32(2)), F32(0))
        v_tl = max(F32(centre[1] - f_dv / F32(2)), F32(0))
        width = min(f_du, F32(wf - u_tl))
        height = min(f_dv, F32(hf - v_tl))
        if not all(math.isfinite(float(x)) for x in (u_tl, v_tl, width, height)):
            status = ST_EPI_POOL_EMPTY
            continue
        rx, ry, rw, rh = int(u_tl), int(v_tl), int(width), int(height)         # cv::Rect(float...) truncates
        if rw <= 0 or rh <= 0 or rx + rw > w or ry + rh > h:
            status = ST_EPI_POOL_EMPTY
            continue
        local = [(F32(a - u_tl), F32(b - v_tl)) for a, b in pool]
        keep, desc = brief32(img[ry:ry + rh, rx:rx + rw], local)
        if len(keep) == 0:
            status = ST_EPI_POOL_EMPTY
            continue
        idx, dist = match_hamming(np.asarray(last_desc, np.uint8), desc)
        if not (p.cutoff_stage3 > dist):
            status = ST_EPI_DIST
            continue
        if not (p.cutoff_original > hamming(np.asarray(orig_desc, np.uint8), desc[idx])):
            status = ST_EPI_ORIG_DIST
            continue
        k = local[keep[idx]]
        return dict(status=ST_OK, uv=(F32(k[0] + u_tl), F32(k[1] + v_tl)), desc=desc[idx].copy())
    return dict(status=status)


def track_stage3(img_l, img_r, tri: Triangulator, T_w2l, lm, motion_scaling: float):
    """Stage 3 for one landmark dict with the extra keys uv_ref (first LEFT detection), ref_desc_l
    (matDescriptorReferenceLEFT) and T_det_l2w (pose of its detection point)."""
    plan = epipolar_plan(tri, T_w2l, lm["T_det_l2w"], lm["uv_ref"], lm["xyz_w"], motion_scaling)
    if plan["status"] != ST_OK:
        return dict(status=plan["status"], stage=0)
    m = epipolar_match(img_l, tri, plan, lm["size"], lm["last_desc_l"], lm["ref_desc_l"])
    if m["status"] != ST_OK:
        return dict(status=m["status"], stage=0)
    size = F32(lm["size"])
    search = F32((1.0 + motion_scaling) * float(F32(lm["last_disparity"])))    # :2415 double product, then float
    x, y = m["uv"]
    r = tri.triangulate_right(img_r, max(F32(0), F32(F32(x - search) - F32(4) * size)), F32(y - F32(4) * size), size, (x, y), m["desc"])
    if r["status"] != ST_OK:
        return dict(status=r["status"], stage=0)
    z = r["xyz"][2]
    if tri.depth_min > z or tri.depth_max < z:
        return dict(status=ST_TRK_DEPTH, stage=0)
    return dict(status=ST_OK, stage=5, uv_l=(x, y), uv_r=r["uv"], xyz=r["xyz"], desc_l=m["desc"], desc_r=r["desc"])


def track_manual_full(img_l, img_r, tri: Triangulator, T_w2l, landmarks, motion_scaling: float):
    """The whole cascade: stages 1, 2 (track_manual) and 3; stage code 5 = stage 3."""
    out = track_manual(img_l, img_r, tri, T_w2l, landmarks, motion_scaling)
    for i, (lm, r) in enumerate(zip(landmarks, out)):
        if r["stage"] or r["status"] == ST_TRK_OUT_OF_FOV or "T_det_l2w" not in lm:
            continue
        out[i] = track_stage3(img_l, img_r, tri, T_w2l, lm, motion_scaling)
    return out


def track_stages(img_l, img_r, tri: Triangulator, T_w2l, landmarks, motion_scaling: float, stages: int):
    """svi_track_landmarks_stages: bit 0 = stage 1, bit 1 = stage 2, bit 2 = stage 3.  Stage 3 alone is the
    moved-camera branch of trackEpipolar (:828-1020): no field-of-view gate in front of it."""
    if stages & 3:
        out = track_manual(img_l, img_r, tri, T_w2l, landmarks, motion_scaling, stage1=bool(stages & 1)) if stages & 2 else \
            track_stage1(img_l, img_r, tri, T_w2l, landmarks, motion_scaling)
    else:
        out = [dict(status=ST_TRK_STAGE1_DIST, stage=0) for _ in landmarks]
    if stages & 4:
        for i, (lm, r) in enumerate(zip(landmarks, out)):
            if r["stage"] or r["status"] == ST_TRK_OUT_OF_FOV:
                continue
            out[i] = track_stage3(img_l, img_r, tri, T_w2l, lm, motion_scaling)
    return out


# ----------------------------------------------------------------------------- CSolverStereoPosit
def transformation_from_vector(v):
    """CMiniVisionToolbox::getTransformationFromVector (src/vision/CMiniVisionToolbox.cpp:354-377): translation
    v[0:3]; rotation = unit quaternion (sqrt(1-|q|^2), q) with q = v[3:6] when |q|^2 < 1, else identity."""
    T = np.eye(4)
    T[:3, 3] = v[:3]
    x, y, z = v[3:6]
    n2 = x * x + y * y + z * z
    if n2 < 1.0:
        w = math.sqrt(1.0 - n2)
        T[:3, :3] = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                              [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                              [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
    return T


def solve_stereo_posit(P_l, P_r, T_last, t_imu, T_estimate, matches, min_points=25, min_inliers=15, max_iter=1000,
                       max_err_inlier=10.0, max_err_avg=9.0, max_risk=2.0, delta=1e-5, min_translation=0.001):
    """CSolverStereoPosit::getTransformationWORLDtoLEFT (src/optimization/CSolverStereoPosit.cpp:8-170): robust
    Gauss-Newton on the stereo reprojection error.  matches: list of (xyz_world (3,), uv_l (2,), uv_r (2,)).
    Returns (T_world_to_left 4x4, None) or (None, reason)."""
    n = len(matches)
    if not (min_points < n):
        return None, "insufficient number of points"
    P_l, P_r = np.asarray(P_l, np.float64).reshape(3, 4), np.asarray(P_r, np.float64).reshape(3, 4)
    T = np.array(T_estimate, np.float64).reshape(4, 4).copy()
    prev = 0.0
    for _ in range(max_iter):
        H = np.zeros((6, 6))
        b = np.zeros(6)
        total = 0.0
        inliers = 0
        for xyz_w, uvl, uvr in matches:
            p = T[:3, :3] @ np.asarray(xyz_w, np.float64) + T[:3, 3]
            if not (0.0 < p[2]):
                continue
            ph = np.append(p, 1.0)
            a_l, a_r = P_l @ ph, P_r @ ph
            cl, cr = a_l[2], a_r[2]
            e = np.array([a_l[0] / cl - float(uvl[0]), a_l[1] / cl - float(uvl[1]), a_r[0] / cr - float(uvr[0]), a_r[1] / cr - float(uvr[1])])
            e2 = float(e @ e)
            w = 1.0
            if max_err_inlier < e2:
                w = max_err_inlier / e2
            else:
                inliers += 1
            total += w * e2
            Jt = np.zeros((4, 6))
            Jt[:3, :3] = np.eye(3)
            Jt[:3, 3:] = -2.0 * np.array([[0, -p[2], p[1]], [p[2], 0, -p[0]], [-p[1], p[0], 0]])
            Jl = np.array([[1 / cl, 0, -a_l[0] / (cl * cl)], [0, 1 / cl, -a_l[1] / (cl * cl)]])
            Jr = np.array([[1 / cr, 0, -a_r[0] / (cr * cr)], [0, 1 / cr, -a_r[1] / (cr * cr)]])
            J = np.vstack([Jl @ P_l @ Jt, Jr @ P_r @ Jt])
            H += w * (J.T @ J)
            b += w * (J.T @ e)
        T = transformation_from_vector(np.linalg.solve(H, -b)) @ T
        R = T[:3, :3].copy()
        RtR = R.T @ R
        RtR[np.diag_indices(3)] -= 1.0
        T[:3, :3] = R - 0.5 * R @ RtR
        if delta > abs(prev - total):
            if max_err_avg < total / n and min_inliers > inliers:
                return None, "insufficient accuracy"
            T_last = np.asarray(T_last, np.float64).reshape(4, 4)
            d = T[:3, 3] - T_last[:3, 3]
            if min_translation > float(d @ d):
                T[:3, 3] = T_last[:3, 3]
            Tinv = np.eye(4)
            Tinv[:3, :3] = T[:3, :3].T
            Tinv[:3, 3] = -T[:3, :3].T @ T[:3, 3]
            Te = np.asarray(T_estimate, np.float64).reshape(4, 4)
            te_inv = -Te[:3, :3].T @ Te[:3, 3]
            r = Tinv[:3, 3] - te_inv - np.asarray(t_imu, np.float64)
            if max_risk < float(r @ r):
                return None, "inconsistent with prior"
            return T, None
        prev = total
    return None, "system did not converge"


# ----------------------------------------------------------------------------- CLandmark::optimize
def optimize_landmark(xyz0, measurements, min_measurements=5, max_iter=1000, delta=1e-5, kernel=10.0, max_avg=9.0, min_ratio=0.5):
    """CLandmark::optimize / _getOptimizedLandmarkSTEREOUV (src/types/CLandmark.cpp:281-296, :447-581).
    measurements: list of (P_world_to_left 3x4, P_world_to_right 3x4, uv_l, uv_r).
    Returns dict(xyz, optimal, success, failed): success / failed are the increments of uOptimizationsSuccessful / Failed."""
    xyz0 = np.asarray(xyz0, np.float64)
    n = len(measurements)
    if not (min_measurements < n):
        return dict(xyz=xyz0, optimal=True, success=0, failed=0)
    X = np.append(xyz0, 1.0)
    prev = 0.0
    for _ in range(max_iter):
        H = np.zeros((4, 4))
        b = np.zeros(4)
        total = 0.0
        inliers = 0
        for P_l, P_r, uvl, uvr in measurements:
            P_l, P_r = np.asarray(P_l, np.float64).reshape(3, 4), np.asarray(P_r, np.float64).reshape(3, 4)
            a_l, a_r = P_l @ X, P_r @ X
            cl, cr = a_l[2], a_r[2]
            e = np.array([a_l[0] / cl - float(uvl[0]), a_l[1] / cl - float(uvl[1]), a_r[0] / cr - float(uvr[0]), a_r[1] / cr - float(uvr[1])])
            e2 = float(e @ e)
            w = 1.0
            if kernel < e2:
                w = kernel / e2
            else:
                inliers += 1
            total += w * e2
            Jl = np.array([[1 / cl, 0, -a_l[0] / (cl * cl)], [0, 1 / cl, -a_l[1] / (cl * cl)]])
            Jr = np.array([[1 / cr, 0, -a_r[0] / (cr * cr)], [0, 1 / cr, -a_r[1] / (cr * cr)]])
            J = np.vstack([Jl @ P_l, Jr @ P_r])
            H += w * (J.T @ J)
            b += w * (J.T @ e)
        X[:3] += np.linalg.lstsq(H[:, :3], -b, rcond=None)[0]
        if delta > abs(prev - total):
            avg = total / n
            if min_ratio < inliers / n:
                return dict(xyz=X[:3].copy(), optimal=bool(max_avg > avg), success=1, failed=0, avg=avg)
            return dict(xyz=xyz0, optimal=False, success=0, failed=1)
        prev = total
    return dict(xyz=xyz0, optimal=False, success=0, failed=1)

