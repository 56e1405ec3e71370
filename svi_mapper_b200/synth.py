"""Deterministic synthetic KITTI-shaped stereo pairs (SURVEY.md section 8(d)).

LEFT  = multi-octave value noise (three Gaussian-blurred uniform-noise layers), u8.
RIGHT = LEFT shifted by a piecewise-constant integer disparity field in 1..55 px
        (xR = xL - d) plus independent +-2 grey-level noise, so most left corners have a
        true match inside the reference's 60 px scan-line search range
        (CTriangulator.h:20 fMinimumSearchRangePixels).

No high-contrast shapes on purpose: they raise max(R) and the 1 % GFTT quality threshold
then removes the texture corners (measured in SURVEY.md section 8(d)).

`stereo_pair` (numpy + cv2, seeded) is the generator used by tests and golden fixtures.
`stereo_batch_torch` builds a large batch directly on the GPU for bench.py.
"""
from __future__ import annotations

import numpy as np

# image sizes of the configurations in BASELINE.md section 4
SIZES = {
    "kitti_00": (1241, 376),
    "kitti_11_12": (1226, 370),
    "vi_sensor": (752, 480),
    "stress": (3840, 1080),
}

_SIGMAS = (1.5, 4.0, 12.0)
_WEIGHTS = (1.0, 0.7, 0.5)


def _minmax(a: np.ndarray) -> np.ndarray:
    lo, hi = float(a.min()), float(a.max())
    return (a - lo) / max(hi - lo, 1e-12)


def left_image(width: int, height: int, seed: int) -> np.ndarray:
    import cv2

    rng = np.random.default_rng(seed)
    acc = np.zeros((height, width), np.float32)
    for sigma, w in zip(_SIGMAS, _WEIGHTS):
        layer = rng.random((height, width), dtype=np.float32)
        layer = cv2.GaussianBlur(layer, (0, 0), sigma)
        acc += np.float32(w) * _minmax(layer).astype(np.float32)
    return np.rint(_minmax(acc) * 255.0).astype(np.uint8)


def disparity_field(width: int, height: int, rng, d_min=1, d_max=55, blocks=(8, 4)) -> np.ndarray:
    """Piecewise-constant integer disparities on the RIGHT image grid."""
    bx, by = blocks
    d_blocks = rng.integers(d_min, d_max + 1, size=(by, bx))
    ys = np.minimum((np.arange(height) * by) // height, by - 1)
    xs = np.minimum((np.arange(width) * bx) // width, bx - 1)
    return d_blocks[ys][:, xs].astype(np.int32)


def right_image(left: np.ndarray, seed: int, d_min=1, d_max=55) -> np.ndarray:
    h, w = left.shape
    rng = np.random.default_rng(seed + 0x5EED)
    d = disparity_field(w, h, rng, d_min, d_max)
    xs = np.arange(w)[None, :] + d  # xL = xR + d
    valid = xs < w
    src = np.take_along_axis(left, np.minimum(xs, w - 1), axis=1)
    fill = rng.integers(0, 256, size=(h, w), dtype=np.int32).astype(np.uint8)
    right = np.where(valid, src, fill).astype(np.int32)
    right += rng.integers(-2, 3, size=(h, w), dtype=np.int32)
    return np.clip(right, 0, 255).astype(np.uint8)


def stereo_pair(width: int, height: int, seed: int, d_min=1, d_max=55):
    """One (left, right) u8 pair, C-contiguous H x W."""
    left = left_image(width, height, seed)
    right = right_image(left, seed, d_min, d_max)
    return np.ascontiguousarray(left), np.ascontiguousarray(right)


def unrectify(img: np.ndarray, cam) -> np.ndarray:
    """The raw image a distorted, unrectified camera would have seen of a rectified image `img` (H, W) u8: every raw pixel
    takes the rectified position cv2.undistortPoints(pixel, K, D, R=R, P=P) of calib.PinholeCamera `cam` and samples `img`
    there bilinearly (0 outside).  For raw test sequences; rectifying the result gives `img` back up to the two
    interpolations."""
    import cv2

    H, W = img.shape
    K = np.asarray(cam.K, np.float64).reshape(3, 3)
    D = np.asarray(cam.distortion, np.float64).reshape(4)
    R = np.asarray(cam.rectification, np.float64).reshape(3, 3)
    P = np.asarray(cam.P, np.float64).reshape(3, 4)
    u, v = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    pts = np.stack([u, v], -1).reshape(-1, 1, 2)
    rect = cv2.undistortPoints(pts, K, D, R=R, P=P).reshape(H, W, 2).astype(np.float32)
    return cv2.remap(img, rect[..., 0], rect[..., 1], cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)


def stereo_batch_torch(n_frames: int, width: int, height: int, seed: int, device="cuda", d_max: int = 55):
    """Batch of n_frames distinct pairs generated on `device` with torch ops.

    Same recipe as stereo_pair (3 blurred noise layers, block disparities 1..55, +-2 noise)
    but with torch's RNG and a separable-convolution blur, so the pixel values differ from
    the numpy generator; every frame of the batch is distinct. Returns two uint8 tensors
    of shape (n_frames, height, width).
    """
    import torch
    import torch.nn.functional as F

    g = torch.Generator(device=device)
    g.manual_seed(seed)
    outs_l, outs_r = [], []
    chunk = 64
    for f0 in range(0, n_frames, chunk):
        n = min(chunk, n_frames - f0)
        acc = torch.zeros((n, 1, height, width), device=device)
        for sigma, wgt in zip(_SIGMAS, _WEIGHTS):
            x = torch.rand((n, 1, height, width), device=device, generator=g)
            r = int(4 * sigma + 0.5)
            t = torch.arange(-r, r + 1, device=device, dtype=torch.float32)
            k = torch.exp(-0.5 * (t / sigma) ** 2)
            k = k / k.sum()
            x = F.conv2d(F.pad(x, (r, r, 0, 0), mode="reflect"), k.view(1, 1, 1, -1))
            x = F.conv2d(F.pad(x, (0, 0, r, r), mode="reflect"), k.view(1, 1, -1, 1))
            lo = x.amin(dim=(2, 3), keepdim=True)
            hi = x.amax(dim=(2, 3), keepdim=True)
            acc += wgt * (x - lo) / (hi - lo)
        lo = acc.amin(dim=(2, 3), keepdim=True)
        hi = acc.amax(dim=(2, 3), keepdim=True)
        left = torch.round((acc - lo) / (hi - lo) * 255.0).to(torch.uint8).squeeze(1)
        by, bx = 4, 8
        d_blocks = torch.randint(1, d_max + 1, (n, by, bx), device=device, generator=g)
        ys = torch.clamp((torch.arange(height, device=device) * by) // height, max=by - 1)
        xs = torch.clamp((torch.arange(width, device=device) * bx) // width, max=bx - 1)
        d = d_blocks[:, ys][:, :, xs]
        src_x = torch.arange(width, device=device).view(1, 1, -1) + d
        valid = src_x < width
        src = torch.gather(left, 2, torch.clamp(src_x, max=width - 1))
        fill = torch.randint(0, 256, (n, height, width), device=device, generator=g).to(torch.uint8)
        right = torch.where(valid, src, fill).to(torch.int16)
        right += torch.randint(-2, 3, (n, height, width), device=device, generator=g).to(torch.int16)
        outs_l.append(left.contiguous())
        outs_r.append(right.clamp_(0, 255).to(torch.uint8).contiguous())
    return torch.cat(outs_l), torch.cat(outs_r)


def stereo_frames_range_torch(first: int, count: int, width: int, height: int, base_seed: int, device="cuda", d_max: int = 55):
    """Frames [first, first + count) of an endless synthetic stream: the stream is generated in blocks (64 frames, 8 for
    multi-megapixel images) with one seeded generator per block, so the content of frame i does not depend on how a batch
    is partitioned over GPUs -- the multi-GPU runs of a fixed batch (BASELINE.json configs[3]) see the same frames as one GPU."""
    import torch

    block = 64 if width * height <= 2_000_000 else 8
    ls, rs = [], []
    if count <= 0:
        e = torch.zeros((0, height, width), dtype=torch.uint8, device=device)
        return e, e.clone()
    for b in range(first // block, (first + count - 1) // block + 1):
        l, r = stereo_batch_torch(block, width, height, seed=base_seed * 1000003 + b, device=device, d_max=d_max)
        lo, hi = max(first, b * block) - b * block, min(first + count, (b + 1) * block) - b * block
        ls.append(l[lo:hi])
        rs.append(r[lo:hi])
    return torch.cat(ls).contiguous(), torch.cat(rs).contiguous()
