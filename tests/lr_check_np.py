"""CPU restatement of the dense left-right check (svi_params.lr_max_diff; include/svi_gpu.h states the rule): the reference's
reverse search, Triangulator.triangulate_left (getPointTriangulatedInLEFT, 7 arguments), from every SVI_OK match of the
oracle's addNewLandmarks, then the sub-pixel refinement of tests/subpixel_np.py on the survivors.  Test and benchmark
infrastructure only, like oracle/."""
from __future__ import annotations

import numpy as np

from oracle import frontend_np as o
import subpixel_np as sp

F32 = np.float32
ST_LR_INCONSISTENT = 27  # dense left-right check (optional mode, no reference text)


def reverse_search(img_l, uv_l, uv_r, desc_r, tri: o.Triangulator, size: float = 7.0) -> dict:
    """The reverse search of one match: getPointTriangulatedInLEFT(img_l, search_range, xR - 4 size, y - 4 size, size,
    (xR, y), desc_r) with y the LEFT key-point's row, corners in fp32."""
    xr, y = F32(uv_r[0]), F32(uv_l[1])
    half = F32(4) * F32(size)
    return tri.triangulate_left(img_l, F32(tri.p.search_range), F32(xr - half), F32(y - half), size, (xr, y), desc_r)


def lr_check(img_l, uv_l, uv_r, desc_r, status, max_diff: int, tri: o.Triangulator, size: float = 7.0) -> np.ndarray:
    """Status after the check: an ST_OK slot stays ST_OK iff its reverse search is ST_OK and lands at most max_diff px (fp32)
    from the LEFT key-point, otherwise it becomes ST_LR_INCONSISTENT; every other slot keeps its status."""
    uv_l, uv_r = np.asarray(uv_l, F32).reshape(-1, 2), np.asarray(uv_r, F32).reshape(-1, 2)
    desc_r = np.asarray(desc_r, np.uint8).reshape(-1, 32)
    status = np.array(status, np.uint8).reshape(-1)
    for i in np.nonzero(status == o.ST_OK)[0]:
        r = reverse_search(img_l, uv_l[i], uv_r[i], desc_r[i], tri, size)
        if not (r["status"] == o.ST_OK and abs(F32(r["uv"][0] - uv_l[i, 0])) <= F32(max_diff)):
            status[i] = ST_LR_INCONSISTENT
    return status


def add_new_landmarks(img_l, img_r, tri: o.Triangulator, mask=None, lr_max_diff: int = -1, subpixel=None) -> dict:
    """The oracle's addNewLandmarks; with lr_max_diff >= 0 the left-right check of its matches (status only); then, with
    subpixel = (w, L), w > 0, the refinement of the slots that are still ST_OK."""
    out = o.add_new_landmarks(img_l, img_r, tri, mask=mask)
    if lr_max_diff >= 0:
        out["status"] = lr_check(img_l, out["uv_l"], out["uv_r"], out["desc_r"], out["status"], lr_max_diff, tri)
    if subpixel is not None and subpixel[0] > 0:
        ok = out["status"] == o.ST_OK
        out["uv_r"], xyz, out["status"] = sp.subpixel_refine(img_l, img_r, out["uv_l"], out["uv_r"], out["status"], subpixel[0], subpixel[1], tri)
        out["xyz"] = np.where((out["status"] == o.ST_OK)[:, None], xyz, out["xyz"])
        out["desc_r"][ok & (out["status"] != o.ST_OK)] = 0
    return out
