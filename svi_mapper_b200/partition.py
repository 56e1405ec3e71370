"""Frame-level data parallelism: stereo pairs are independent (addNewLandmarks keeps no state between pairs and
CTriangulator is const), so a batch is cut into contiguous frame ranges, one per GPU, with no collective on the data
path (SURVEY.md 8e).

  MultiFrontend      the in-library driver (svi_multi_*): one host thread + one svi_ctx per GPU inside ONE process,
                     disjoint slices of the caller's arrays -- what a C++ tracker links against
  frame_range        the same partition for one-process-per-GPU launches (torchrun: bench.py, tests), where every
                     rank owns a StereoFrontend and only the timing is reduced (max over ranks)"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .frontend import StereoFrames, SviError, _cam, _ptr


def frame_range(n_frames: int, world: int, rank: int) -> tuple[int, int]:
    """Contiguous range [g*F/G, (g+1)*F/G) of rank g; ranges are disjoint and cover [0, F)."""
    if world < 1 or not (0 <= rank < world) or n_frames < 0:
        raise ValueError("bad partition arguments")
    return (rank * n_frames) // world, ((rank + 1) * n_frames) // world


def max_over_ranks(value: float, device=None) -> float:
    """Max of a scalar over all ranks of the default process group (identity without one)."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


class MultiFrontend:
    """svi_multi: the new-landmark path of a batch over several GPUs of one box (frame partition, no collective)."""

    def __init__(self, cam_left, cam_right, devices, lib_path=None, **overrides):
        self._lib = _lib.load(lib_path)
        self.params = _lib.Params()
        self._lib.svi_params_default(C.byref(self.params))
        for k, v in overrides.items():
            if not hasattr(self.params, k):
                raise TypeError(f"unknown svi_params field {k!r}")
            setattr(self.params, k, v)
        self.width, self.height, self.max_corners = int(cam_left.width), int(cam_left.height), int(self.params.max_corners)
        self.devices = [int(d) for d in devices]
        dev = (C.c_int32 * len(self.devices))(*self.devices)
        self._m = C.c_void_p()
        cl, cr = _cam(cam_left), _cam(cam_right)
        rc = self._lib.svi_multi_create(C.byref(cl), C.byref(cr), C.byref(self.params), dev, len(self.devices), C.byref(self._m))
        if rc != _lib.SVI_SUCCESS:
            raise SviError(rc, self._lib.svi_multi_last_error(None).decode())

    def close(self):
        if getattr(self, "_m", None) and self._m.value:
            self._lib.svi_multi_destroy(self._m)
            self._m = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_rectification(self, cam_left, cam_right, float_maps: bool = False):
        """svi_multi_set_rectification: StereoFrontend.set_rectification on every context."""
        from .frontend import rectification
        rl, rr = rectification(cam_left, float_maps), rectification(cam_right, float_maps)
        rc = self._lib.svi_multi_set_rectification(self._m, C.byref(rl), C.byref(rr))
        if rc != _lib.SVI_SUCCESS:
            raise SviError(rc, self._lib.svi_multi_last_error(self._m).decode())

    def clear_rectification(self):
        rc = self._lib.svi_multi_set_rectification(self._m, None, None)
        if rc != _lib.SVI_SUCCESS:
            raise SviError(rc, self._lib.svi_multi_last_error(self._m).decode())

    def frame_range(self, n_frames: int, part: int) -> tuple[int, int]:
        a, b = C.c_int32(), C.c_int32()
        rc = self._lib.svi_multi_frame_range(self._m, int(n_frames), int(part), C.byref(a), C.byref(b))
        if rc != _lib.SVI_SUCCESS:
            raise SviError(rc, "svi_multi_frame_range: bad argument")
        return a.value, a.value + b.value

    def stereo_frames_raw(self, left_ptr, right_ptr, pitch, frame_stride, n_frames, result: _lib.StereoResult, masks_ptr=None):
        rc = self._lib.svi_multi_stereo_frames(self._m, left_ptr, right_ptr, pitch, frame_stride, n_frames, masks_ptr, C.byref(result))
        if rc != _lib.SVI_SUCCESS:
            raise SviError(rc, self._lib.svi_multi_last_error(self._m).decode())

    def stereo_frames(self, left, right, masks=None) -> StereoFrames:
        L = np.ascontiguousarray(left, np.uint8)
        R = np.ascontiguousarray(right, np.uint8)
        if L.ndim != 3 or L.shape != R.shape or L.shape[1:] != (self.height, self.width):
            raise ValueError(f"expected two (n, {self.height}, {self.width}) uint8 batches")
        M = np.ascontiguousarray(masks, np.uint8) if masks is not None else None
        n, cap = L.shape[0], self.max_corners
        out = StereoFrames(
            n_keypoints=np.zeros(n, np.int32), n_detected=np.zeros(n, np.int32),
            uv_left=np.zeros((n, cap, 2), np.float32), uv_right=np.zeros((n, cap, 2), np.float32),
            xyz_left=np.zeros((n, cap, 3), np.float64), desc_left=np.zeros((n, cap, 32), np.uint8),
            desc_right=np.zeros((n, cap, 32), np.uint8), distance=np.full((n, cap), -1, np.int32),
            match_index=np.full((n, cap), -1, np.int32), status=np.zeros((n, cap), np.uint8))
        r = _lib.StereoResult(cap, _ptr(out.n_keypoints), _ptr(out.n_detected), _ptr(out.uv_left), _ptr(out.uv_right),
                              _ptr(out.xyz_left), _ptr(out.desc_left), _ptr(out.desc_right), _ptr(out.distance),
                              _ptr(out.match_index), _ptr(out.status))
        self.stereo_frames_raw(_ptr(L), _ptr(R), self.width, self.width * self.height, n, r, _ptr(M))
        return out
