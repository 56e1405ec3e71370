"""CPU restatement of the sub-pixel disparity mode (svi_params.subpixel_window / subpixel_search; include/svi_gpu.h states the
steps): ORB-SLAM2's Frame::ComputeStereoMatches refinement on top of the oracle's integer-disparity results.  Test and
benchmark infrastructure only, like oracle/."""
from __future__ import annotations

import numpy as np

from oracle import frontend_np as o

F32 = np.float32
ST_SPARSE_NOT_MUTUAL = 25  # sparse frames, left-right check (optional mode, no reference text)
ST_SUBPIXEL_REJECTED = 26  # sub-pixel refinement: the SAD minimum lies on the edge of the search (optional mode, no reference text)


def subpixel_refine(img_l, img_r, uv_l, uv_r, status, w: int, L: int, tri: o.Triangulator):
    """Every ST_OK slot's integer match refined by the first strict SAD minimum of the centred (2w+1)^2 patches over the
    offsets -L..L on the LEFT row and a parabola through its neighbours (fp32), then getPointInLEFT again.  Returns new
    (uv_r, xyz, status) arrays; xyz is zero where the refined status is not ST_OK, uv_r keeps its input there."""
    uv_l, uv_r = np.asarray(uv_l, F32).reshape(-1, 2), np.array(uv_r, F32).reshape(-1, 2)
    status = np.array(status, np.uint8).reshape(-1)
    xyz = np.zeros((len(status), 3), np.float64)
    H, W = img_l.shape
    il, ir = img_l.astype(np.int32), img_r.astype(np.int32)
    for i in np.nonzero(status == o.ST_OK)[0]:
        xl, y, xr = int(uv_l[i, 0]), int(uv_l[i, 1]), int(uv_r[i, 0])
        if xr - w - L < 0 or xr + w + L >= W or xl - w < 0 or xl + w >= W or y - w < 0 or y + w >= H:
            status[i] = ST_SUBPIXEL_REJECTED
            continue
        pl = il[y - w:y + w + 1, xl - w:xl + w + 1]
        pl = pl - pl[w, w]
        sad = []
        for k in range(-L, L + 1):
            pr = ir[y - w:y + w + 1, xr + k - w:xr + k + w + 1]
            sad.append(int(np.abs(pl - (pr - pr[w, w])).sum()))
        j = int(np.argmin(sad))            # the first minimum
        if j == 0 or j == 2 * L:
            status[i] = ST_SUBPIXEL_REJECTED
            continue
        s1, s2, s3 = sad[j - 1], sad[j], sad[j + 1]
        delta = F32(s1 - s3) / (F32(2) * F32(s1 + s3 - 2 * s2))
        x_new = F32(F32(uv_r[i, 0] + F32(j - L)) + delta)
        st, p = tri.point_in_left(uv_l[i], (x_new, uv_r[i, 1]))
        status[i] = st
        if st == o.ST_OK:
            uv_r[i, 0], xyz[i] = x_new, p
    return uv_r, xyz, status


def add_new_landmarks(img_l, img_r, tri: o.Triangulator, mask=None, subpixel=None) -> dict:
    """The oracle's addNewLandmarks, then, with subpixel = (w, L), w > 0, the refinement of its matches."""
    out = o.add_new_landmarks(img_l, img_r, tri, mask=mask)
    if subpixel is not None and subpixel[0] > 0:
        ok = out["status"] == o.ST_OK
        out["uv_r"], xyz, out["status"] = subpixel_refine(img_l, img_r, out["uv_l"], out["uv_r"], out["status"], subpixel[0], subpixel[1], tri)
        out["xyz"] = np.where((out["status"] == o.ST_OK)[:, None], xyz, out["xyz"])
        out["desc_r"][ok & (out["status"] != o.ST_OK)] = 0
    return out
