"""Caller images reach the device through one staging path (DESIGN.md section 3): page-locked memory is read in place, pageable
memory of the single-pair and single-image calls is packed into the pinned image mirror, everything else is copied straight
from the caller.  Every image entry point gets the same content as pageable dense rows, as pageable rows with a padded pitch
and frame stride (garbage in the padding), and as both of these in page-locked memory; the results must equal the pageable
dense ones byte for byte -- with rectification off (kitti_00) and on (vi_sensor), on a context of 4-frame chunks so that the
5-frame calls cross a chunk boundary."""
import ctypes as C
import pathlib

import numpy as np
import pytest

from svi_mapper_b200 import StereoFrontend, load_camera
from svi_mapper_b200.frontend import StereoFrames
from svi_mapper_b200.synth import stereo_pair

CALIB = pathlib.Path(__file__).resolve().parent / "golden" / "calib"

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("built_library")]

CHUNK = 4
FORMS = ("pageable padded", "pinned dense", "pinned padded")

# per entry point: positions of the image arguments, of the pitch, of the frame stride and of the frame count (None: one frame)
IMAGE_ARGS = {
    "svi_harris_response": ((1,), 2, None, None),
    "svi_detect": ((1, 5), 2, 3, 4),
    "svi_describe": ((1,), 2, None, None),
    "svi_triangulate_right": ((1,), 2, None, None),
    "svi_triangulate_left": ((1,), 2, None, None),
    "svi_stereo_frames": ((1, 2, 6), 3, 4, 5),
    "svi_stereo_frame_masked": ((1, 2), 3, None, None),
    "svi_stereo_frames_sparse": ((1, 2, 6), 3, 4, 5),
    "svi_track_landmarks": ((1, 2), 3, None, None),
    "svi_track_frame_stereo_only": ((1, 2), 3, None, None),
    "svi_rectify": ((2,), 3, 4, 5),
}


class Relayout:
    """Stands in for StereoFrontend._lib: the dense image arguments the wrappers pass to the entry points above are copied into
    the memory form `form` (pitch W + 13 and H + 2 rows per frame when padded) before the call."""

    def __init__(self, lib, form, W, H):
        self._lib, self._form, self._W, self._H = lib, form, W, H
        self._rng = np.random.default_rng(17)

    def _buffer(self, nf):
        padded = self._form.endswith("padded")
        shape = (nf, self._H + 2, self._W + 13) if padded else (nf, self._H, self._W)
        if self._form.startswith("pinned"):
            import torch
            buf = torch.empty(shape, dtype=torch.uint8).pin_memory()
            a = buf.numpy()
        else:
            buf = a = np.empty(shape, np.uint8)
        a[...] = self._rng.integers(0, 256, shape, dtype=np.uint8)
        return buf, a

    def __getattr__(self, name):
        f = getattr(self._lib, name)
        if name not in IMAGE_ARGS:
            return f
        images, i_pitch, i_stride, i_frames = IMAGE_ARGS[name]
        W, H = self._W, self._H

        def call(*args):
            args = list(args)
            nf = 1 if i_frames is None else int(args[i_frames])
            keep = []
            for i in images:
                if args[i] is None:
                    continue
                src = np.ctypeslib.as_array((C.c_uint8 * (nf * H * W)).from_address(args[i])).reshape(nf, H, W)
                buf, a = self._buffer(nf)
                a[:, :H, :W] = src
                keep.append(buf)
                args[i] = a.ctypes.data
                args[i_pitch] = a.shape[2]
                if i_stride is not None:
                    args[i_stride] = a.shape[1] * a.shape[2]
            return f(*args)
        return call


def _flat(r):
    """Every array of a result as bytes; in a stereo frame the RIGHT-side fields of a key-point without a match are unspecified."""
    if isinstance(r, StereoFrames):
        return _flat([r.frame(k) for k in range(len(r.n_keypoints))]) + [r.n_detected.tobytes()]
    if isinstance(r, dict):
        ok = r["status"] == 0 if "idx" in r else None
        return [b for k in sorted(r) for b in _flat(r[k][ok] if ok is not None and k in ("uv_r", "xyz", "desc_r") else r[k])]
    if isinstance(r, (list, tuple)):
        return [b for v in r for b in _flat(v)]
    if isinstance(r, np.ndarray):
        return [r.tobytes()]
    return [repr(r).encode()]


@pytest.fixture(scope="module", params=["kitti_00", "vi_sensor rectified"])
def setup(request):
    name = request.param.split()[0]
    cams = load_camera(str(CALIB / f"{name}_left.txt")), load_camera(str(CALIB / f"{name}_right.txt"))
    W, H = cams[0].width, cams[0].height
    pairs = [stereo_pair(W, H, 2600 + i) for i in range(CHUNK + 1)]
    L, R = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    rng = np.random.default_rng(23)
    M = np.full((CHUNK + 1, H, W), 255, np.uint8)
    for f in range(CHUNK + 1):
        for x, y in zip(rng.integers(0, W - 40, 30), rng.integers(0, H - 40, 30)):
            M[f, y:y + 40, x:x + 40] = 0
    with StereoFrontend(*cams, chunk_frames=CHUNK) as fe:
        if request.param.endswith("rectified"):
            fe.set_rectification(*cams)
        n = 200
        xy = np.stack([rng.integers(28, W - 28, n), rng.integers(28, H - 28, n)], 1).astype(np.float32)
        desc_l, _ = fe.describe(L[0], xy)
        desc_r, _ = fe.describe(R[0], xy)
        search = rng.uniform(0.5, 90.0, n).astype(np.float32)
        f0 = fe.stereo_frames(L[0], R[0]).frame(0)
        ok = np.flatnonzero(f0["status"] == 0)[:400]
        assert len(ok) > 50
        T_det = np.broadcast_to(np.eye(4), (len(ok), 4, 4)).copy()
        T_det[::2, 0, 3] = 0.1   # half of the landmarks moved since detection: stage 3 has work too
        lm = dict(xyz=f0["xyz"][ok], dl=f0["desc_l"][ok], dr=f0["desc_r"][ok], disp=(f0["uv_l"][ok, 0] - f0["uv_r"][ok, 0]).astype(np.float32),
                  uv_ref=f0["uv_l"][ok], T_det=T_det)
        L1, R1 = np.roll(L[0], (1, 2), axis=(0, 1)), np.roll(R[0], (1, 2), axis=(0, 1))   # stage 2 has work too
        yield fe, dict(L=L, R=R, M=M, xy=xy, desc_l=desc_l, desc_r=desc_r, search=search, lm=lm, L1=L1, R1=R1,
                       rect=request.param.endswith("rectified"))


ENTRIES = {
    "harris_response": lambda fe, d: fe.harris_response(d["L"][0]),
    "detect 1 frame": lambda fe, d: fe.detect(d["L"][:1], d["M"][:1]),
    "detect chunk + 1 frames": lambda fe, d: fe.detect(d["L"], d["M"]),
    "describe": lambda fe, d: fe.describe(d["L"][0], d["xy"]),
    "triangulate_right": lambda fe, d: fe.triangulate_right(
        d["R"][0], np.stack([np.maximum(0, d["xy"][:, 0] - 28 - d["search"]), d["xy"][:, 1] - 28], 1).astype(np.float32), d["xy"], d["desc_l"]),
    "triangulate_left": lambda fe, d: fe.triangulate_left(d["L"][0], d["search"], d["xy"] - np.float32(28), d["xy"], d["desc_r"]),
    "stereo_frames 1 pair": lambda fe, d: fe.stereo_frames(d["L"][:1], d["R"][:1], d["M"][:1]),
    "stereo_frames 2 pairs": lambda fe, d: fe.stereo_frames(d["L"][:2], d["R"][:2], d["M"][:2]),
    "stereo_frames chunk + 1 pairs": lambda fe, d: fe.stereo_frames(d["L"], d["R"], d["M"]),
    "stereo_frame_masked": lambda fe, d: fe.add_new_landmarks(d["L"][1], d["R"][1], mask_centres=d["xy"]),
    "stereo_frames_sparse mutual": lambda fe, d: fe.stereo_frames_sparse(d["L"], d["R"], d["M"], mutual=True),
    "track_landmarks": lambda fe, d: fe.track_landmarks(
        d["L1"], d["R1"], np.eye(4), d["lm"]["xyz"], d["lm"]["dl"], d["lm"]["dr"], d["lm"]["disp"], 7.0, 1.0,
        uv_reference_left=d["lm"]["uv_ref"], desc_reference_left=d["lm"]["dl"], T_left_to_world_at_detection=d["lm"]["T_det"]),
    "track_frame_stereo_only": lambda fe, d: fe.track_frame_stereo_only(
        d["L1"], d["R1"], d["lm"]["xyz"], d["lm"]["dl"], d["lm"]["dr"], d["lm"]["disp"], 7.0, d["lm"]["uv_ref"], d["lm"]["dl"],
        d["lm"]["T_det"], np.ones(len(d["lm"]["xyz"]), np.uint8), np.eye(4), np.eye(4), np.eye(4), np.zeros(3), 1.0),
    "rectify": lambda fe, d: fe.rectify(d["R"], 1),
}


@pytest.mark.parametrize("entry", list(ENTRIES))
def test_every_memory_form_gives_the_same_result(setup, entry):
    fe, d = setup
    if entry == "rectify" and not d["rect"]:
        pytest.skip("svi_rectify needs a rectification")
    lib = fe._lib
    want = _flat(ENTRIES[entry](fe, d))
    for form in FORMS:
        fe._lib = Relayout(lib, form, fe.width, fe.height)
        try:
            got = _flat(ENTRIES[entry](fe, d))
        finally:
            fe._lib = lib
        assert got == want, form
