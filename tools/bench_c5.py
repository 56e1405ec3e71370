#!/usr/bin/env python3
"""Sparse stereo frames (svi_stereo_frames_sparse) on a B200; prints one JSON object (--out: also writes it there).

  c5     one 3840 x 1080 pair, maxCorners 10000 (BASELINE.json C5): the fused sparse call against the composed four-call
         chain it replaces (detect both images, describe both, match_epipolar), outputs compared byte for byte first, at a
         +-1 row band (disparity 1..1000) and at a brute-force band; the dense scan-line frame (range 1000 px) beside it
  batch  device-resident batches, sparse vs dense frames/s: 16 C5 frames, and a C2-shaped batch (4096 x 1241 x 376, K 2000)
  kernel band_match_kernel's time from torch.profiler (a separate run), the algorithmic popc count (8 x the admissible pairs,
         counted on the host from the key-point lists) and its share of 148 SMs x 16 popc per clock at the card's SM clock
The card's name, power limit and SM clock are read in the same run."""
import argparse
import json
import pathlib
import subprocess
import sys
import time
from types import SimpleNamespace

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from svi_mapper_b200 import StereoFrontend, _lib, load_camera  # noqa: E402
from svi_mapper_b200.synth import stereo_pair  # noqa: E402

W5, H5, K5, RANGE5 = 3840, 1080, 10000, 1000.0
BANDS = {"band_pm1": (1.0, 1.0, RANGE5), "brute_force": (1e9, -1e9, 1e9)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, pl, sm, smax = (s.strip() for s in q.split(","))
    return dict(name=name, power_limit_w=float(pl), sm_clock_mhz=float(sm), sm_clock_max_mhz=float(smax))


def median_ms(fn, reps, warm=2):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts) * 1e3)


def kitti():
    calib = ROOT / "tests" / "golden" / "calib"
    return load_camera(str(calib / "kitti_00_left.txt")), load_camera(str(calib / "kitti_00_right.txt"))


def admissible_pairs(kl, kr, band):
    """Pairs |yL - yR| <= band_v, dmin <= xL - xR <= dmax, counted row by row on the host (fp32 tests as in the kernel)."""
    kl, kr = kl.astype(np.float32), kr.astype(np.float32)
    total = 0
    for i in range(0, len(kl), 512):
        q = kl[i:i + 512]
        d = q[:, None, 0] - kr[None, :, 0]
        total += int(((np.abs(q[:, None, 1] - kr[None, :, 1]) <= np.float32(band[0])) & (d >= np.float32(band[1])) &
                      (d <= np.float32(band[2]))).sum())
    return total


def bench_c5(out, reps):
    from test_sparse_frames import assert_same, composed_np
    k0, k1 = kitti()
    cl, cr = SimpleNamespace(width=W5, height=H5, P=k0.P), SimpleNamespace(width=W5, height=H5, P=k1.P)
    L, R = stereo_pair(W5, H5, 3000, d_max=900)
    with StereoFrontend(cl, cr, max_corners=K5, search_range_px=RANGE5, max_candidates=131072, chunk_frames=1) as fe:
        res = {}
        for name, band in BANDS.items():
            fused = fe.stereo_frames_sparse(L, R, None, *band).frame(0)
            comp = composed_np(fe, L, R, band)
            assert_same(fused, comp, name)   # byte for byte before any timing
            kr = fe.detect(R)[0]
            kr = kr[fe.describe(R, kr)[1]]
            res[name] = dict(band=band, left_keypoints=len(fused["uv_l"]), right_keypoints=int(fused["n_right"]),
                             matched=int((fused["status"] == 0).sum()), identical_to_composed=True,
                             admissible_pairs=admissible_pairs(fused["uv_l"], kr, band),
                             fused_ms=median_ms(lambda: fe.stereo_frames_sparse(L, R, None, *band), reps),
                             composed_ms=median_ms(lambda: composed_np(fe, L, R, band), reps))
        res["dense_ms"] = median_ms(lambda: fe.stereo_frames(L, R), reps)
    out["c5"] = res


def device_batch(cams, n, pair_seeds, params, band, reps):
    """Device-resident batch: frames/s of stereo_frames_device and stereo_frames_sparse_device (events around `reps` calls)."""
    import torch
    W, H = cams[0].width, cams[0].height
    base = [stereo_pair(W, H, s, **pair_seeds[1]) for s in pair_seeds[0]]
    Ls = torch.from_numpy(np.stack([base[i % len(base)][0] for i in range(n)])).cuda()
    Rs = torch.from_numpy(np.stack([base[i % len(base)][1] for i in range(n)])).cuda()
    with StereoFrontend(*cams, **params) as fe:
        cap = fe.max_corners
        from svi_mapper_b200.frontend import StereoFrames
        host = StereoFrames.empty(1, 1, sparse=True)
        dev = {k: torch.zeros((n,) + v.shape[1:2] if v.ndim == 1 else (n, cap) + v.shape[2:], dtype=torch.from_numpy(v).dtype, device="cuda")
               for k, v in vars(host).items()}
        r = _lib.StereoResult(cap, *[dev[k].data_ptr() for k in ("n_keypoints", "n_detected", "uv_left", "uv_right", "xyz_left", "desc_left",
                                                                  "desc_right", "distance", "match_index", "status")])
        sp = _lib.SparseResult(dev["second_distance"].data_ptr(), dev["n_keypoints_right"].data_ptr())
        stream = torch.cuda.current_stream().cuda_stream
        calls = {"dense": lambda: fe.stereo_frames_device(Ls.data_ptr(), Rs.data_ptr(), W, W * H, n, r, stream=stream),
                 "sparse": lambda: fe.stereo_frames_sparse_device(Ls.data_ptr(), Rs.data_ptr(), W, W * H, n, r, sp, *band, stream=stream)}
        out = {}
        for name, fn in calls.items():
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
            fe.check_overflow()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            fe.check_overflow()
            ms = e0.elapsed_time(e1) / reps
            out[name] = dict(ms_per_call=ms, frames_per_s=n / ms * 1e3)
        out["mean_keypoints"] = dict(left=float(dev["n_keypoints"].float().mean()), right=float(dev["n_keypoints_right"].float().mean()))
    return out


def bench_batch(out, reps):
    k0, k1 = kitti()
    c5 = (SimpleNamespace(width=W5, height=H5, P=k0.P), SimpleNamespace(width=W5, height=H5, P=k1.P))
    out["batch"] = {
        "c5_x16": dict(band=BANDS["band_pm1"], **device_batch(c5, 16, ([3000, 3001], dict(d_max=900)),
                                                              dict(max_corners=K5, search_range_px=RANGE5, max_candidates=131072),
                                                              BANDS["band_pm1"], reps)),
        "c2_x4096": dict(band=(1.0, 1.0, 60.0), **device_batch(kitti(), 4096, (list(range(1000, 1016)), {}), dict(max_corners=2000),
                                                                (1.0, 1.0, 60.0), reps)),
    }


def bench_kernel(out, clock_mhz):
    """band_match_kernel's device time per C5 frame from torch.profiler, against 8 popc per admissible pair."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    k0, k1 = kitti()
    cl, cr = SimpleNamespace(width=W5, height=H5, P=k0.P), SimpleNamespace(width=W5, height=H5, P=k1.P)
    L, R = stereo_pair(W5, H5, 3000, d_max=900)
    res = {}
    with StereoFrontend(cl, cr, max_corners=K5, search_range_px=RANGE5, max_candidates=131072, chunk_frames=1) as fe:
        for name, band in BANDS.items():
            fe.stereo_frames_sparse(L, R, None, *band)
            reps = 10
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    fe.stereo_frames_sparse(L, R, None, *band)
                torch.cuda.synchronize()
            us = [e.device_time_total for e in prof.key_averages() if "band_match_kernel" in e.key]
            kernel_us = sum(us) / reps
            pairs = out["c5"][name]["admissible_pairs"]
            popc = 8 * pairs
            ideal_us = popc / (148 * 16 * clock_mhz * 1e6) * 1e6
            res[name] = dict(kernel_us=kernel_us, admissible_pairs=pairs, popc=popc, popc_bound_us=ideal_us,
                             share_of_popc_peak=ideal_us / kernel_us if kernel_us else None)
    out["band_match_kernel"] = res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"card": card()}
    bench_c5(out, a.reps)
    bench_batch(out, a.reps)
    bench_kernel(out, out["card"]["sm_clock_max_mhz"])
    out["card_after"] = card()
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        pathlib.Path(a.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
