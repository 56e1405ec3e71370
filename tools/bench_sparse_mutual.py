#!/usr/bin/env python3
"""The left-right check of sparse stereo frames (svi_sparse_band.mutual) on a B200; prints one JSON object (--out: also
writes it there).

  c5         the C5 pair (3840 x 1080, maxCorners 10000) at a +-1 row band and at a brute-force band: the fused call with and
             without the check, each output first compared byte for byte with the composed public calls; medians of
             synchronous calls, the two runs alternated; the precision of the accepted matches against the true disparity
  kernel     torch.profiler (a separate run): band_match_kernel's forward and reverse passes and gather_rows_kernel per C5 frame
  batch      device-resident batches (16 C5 frames, 4096 x 1241 x 376): frames/s with and without the check, alternated
  --ab LIB   the check-off path against another build of the library (SVI_GPU_LIB), alternated A B A B in fresh processes:
             tools/bench_c5.py's sparse batch lines and bench.py --config c5's value
The card's name, power limit and SM clock are read in the same run."""
import argparse
import json
import os
import pathlib
import subprocess
import sys
import time
from types import SimpleNamespace

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))

from bench_c5 import BANDS, H5, K5, RANGE5, W5, card, kitti  # noqa: E402
from svi_mapper_b200 import StereoFrontend, _lib  # noqa: E402
from svi_mapper_b200.synth import disparity_field, stereo_pair  # noqa: E402

SEED5, DMAX5 = 3000, 900
REJECTED = (_lib.SVI_TRI_NO_MATCH, _lib.SVI_TRI_DISTANCE, _lib.SVI_SPARSE_NOT_MUTUAL)


def c5_frontend():
    k0, k1 = kitti()
    cams = SimpleNamespace(width=W5, height=H5, P=k0.P), SimpleNamespace(width=W5, height=H5, P=k1.P)
    return StereoFrontend(*cams, max_corners=K5, search_range_px=RANGE5, max_candidates=131072, chunk_frames=1)


def precision(frame, kr, d_true):
    """Accepted slots (not rejected by the cut-off or the check) and how many of them are right: same row and
    |x_L - x_R - d_true(x_R, y)| <= 1."""
    acc = ~np.isin(frame["status"], REJECTED)
    kl, j = frame["uv_l"][acc].astype(np.int64), frame["idx"][acc]
    r = kr[j].astype(np.int64)
    good = (r[:, 1] == kl[:, 1]) & (np.abs(kl[:, 0] - r[:, 0] - d_true[r[:, 1], r[:, 0]]) <= 1)
    return dict(accepted=int(acc.sum()), correct=int(good.sum()), precision=float(good.sum() / max(acc.sum(), 1)))


def bench_c5(out, reps):
    from test_sparse_frames import assert_same, composed_np
    from test_sparse_mutual import _assert_off_on, composed_mutual
    L, R = stereo_pair(W5, H5, SEED5, d_max=DMAX5)
    d_true = disparity_field(W5, H5, np.random.default_rng(SEED5 + 0x5EED), 1, DMAX5)
    res = {}
    with c5_frontend() as fe:
        kr = fe.detect(R)[0]
        kr = kr[fe.describe(R, kr)[1]]
        for name, band in BANDS.items():
            off = fe.stereo_frames_sparse(L, R, None, *band)
            on = fe.stereo_frames_sparse(L, R, None, *band, mutual=True)
            assert_same(off.frame(0), composed_np(fe, L, R, band), name)        # byte for byte before any timing
            assert_same(on.frame(0), composed_mutual(fe, L, R, band), name)
            _assert_off_on(off, on)
            t = {False: [], True: []}
            for m in (False, True, False, True):
                fe.stereo_frames_sparse(L, R, None, *band, mutual=m)
            for _ in range(reps):
                for m in (False, True):
                    t0 = time.perf_counter()
                    fe.stereo_frames_sparse(L, R, None, *band, mutual=m)
                    t[m].append(time.perf_counter() - t0)
            res[name] = dict(band=band, left_keypoints=int(off.n_keypoints[0]), right_keypoints=int(off.n_keypoints_right[0]),
                             identical_to_composed=True, off_ms=float(np.median(t[False]) * 1e3),
                             on_ms=float(np.median(t[True]) * 1e3), reps=reps,
                             not_mutual=int((on.status[0] == _lib.SVI_SPARSE_NOT_MUTUAL).sum()),
                             precision_off=precision(off.frame(0), kr, d_true), precision_on=precision(on.frame(0), kr, d_true))
    out["c5"] = res


def bench_kernel(out):
    """Device time per C5 frame of the forward pass, the reverse pass and the gather, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    L, R = stereo_pair(W5, H5, SEED5, d_max=DMAX5)
    res = {}
    with c5_frontend() as fe:
        for name, band in BANDS.items():
            res[name] = {}
            for m in (False, True):
                fe.stereo_frames_sparse(L, R, None, *band, mutual=m)
                reps = 10
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(reps):
                        fe.stereo_frames_sparse(L, R, None, *band, mutual=m)
                    torch.cuda.synchronize()
                res[name]["on" if m else "off"] = {e.key: e.device_time_total / reps for e in prof.key_averages()
                                                   if "band_match_kernel" in e.key or "gather_rows_kernel" in e.key}
    out["kernels_us_per_frame"] = res


def device_batch(cams, n, pair_seeds, params, band, reps):
    """Device-resident batch: frames/s of stereo_frames_sparse_device without and with the check (events around `reps`
    calls, the two alternated twice)."""
    import torch
    from svi_mapper_b200.frontend import StereoFrames
    W, H = cams[0].width, cams[0].height
    base = [stereo_pair(W, H, s, **pair_seeds[1]) for s in pair_seeds[0]]
    Ls = torch.from_numpy(np.stack([base[i % len(base)][0] for i in range(n)])).cuda()
    Rs = torch.from_numpy(np.stack([base[i % len(base)][1] for i in range(n)])).cuda()
    with StereoFrontend(*cams, **params) as fe:
        cap = fe.max_corners
        host = StereoFrames.empty(1, 1, sparse=True)
        dev = {k: torch.zeros((n,) + v.shape[1:2] if v.ndim == 1 else (n, cap) + v.shape[2:], dtype=torch.from_numpy(v).dtype, device="cuda")
               for k, v in vars(host).items()}
        r = _lib.StereoResult(cap, *[dev[k].data_ptr() for k in ("n_keypoints", "n_detected", "uv_left", "uv_right", "xyz_left", "desc_left",
                                                                  "desc_right", "distance", "match_index", "status")])
        sp = _lib.SparseResult(dev["second_distance"].data_ptr(), dev["n_keypoints_right"].data_ptr())
        stream = torch.cuda.current_stream().cuda_stream

        def call(m):
            fe.stereo_frames_sparse_device(Ls.data_ptr(), Rs.data_ptr(), W, W * H, n, r, sp, *band, stream=stream, mutual=m)
        for m in (False, True):
            for _ in range(2):
                call(m)
        torch.cuda.synchronize()
        fe.check_overflow()
        out = {"off": [], "on": []}
        for m in (False, True, False, True):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                call(m)
            e1.record()
            torch.cuda.synchronize()
            fe.check_overflow()
            out["on" if m else "off"].append(n / (e0.elapsed_time(e1) / reps) * 1e3)
        out = {k: dict(frames_per_s=v, mean_frames_per_s=float(np.mean(v))) for k, v in out.items()}
        out["not_mutual_share"] = float((dev["status"] == _lib.SVI_SPARSE_NOT_MUTUAL).sum() / dev["n_keypoints"].sum())
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


def bench_ab(out, other, reps):
    """The check-off path: this build against `other`, A B A B in fresh processes (the spread of A against A is the noise)."""
    res = {"other_lib": str(other), "order": [], "sparse_batch_fps": {"c5_x16": [], "c2_x4096": []}, "bench_c5_value": []}
    code = ("import json,sys; sys.path.insert(0,'tools'); import bench_c5 as b; o={}; b.bench_batch(o,%d); "
            "print(json.dumps({k: v['sparse']['frames_per_s'] for k, v in o['batch'].items()}))" % reps)
    for lib in ("other", "this", "other", "this"):
        env = dict(os.environ)
        env.pop("SVI_GPU_LIB", None)
        if lib == "other":
            env["SVI_GPU_LIB"] = str(other)
        res["order"].append(lib)
        p = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, check=True)
        fps = json.loads(p.stdout.strip().splitlines()[-1])
        for k in fps:
            res["sparse_batch_fps"][k].append(fps[k])
        p = subprocess.run([sys.executable, "bench.py", "--config", "c5", "--steps", "20", "--warmup", "3", "--no-cpu-baseline"],
                           cwd=ROOT, env=env, capture_output=True, text=True, check=True)
        res["bench_c5_value"].append(json.loads(p.stdout.strip().splitlines()[-1])["value"])
    out["check_off_ab"] = res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--part", default="c5,batch", help="comma list of c5, kernel, batch")
    ap.add_argument("--ab", default=None, metavar="LIB", help="another build of libsvi_gpu.so to compare the check-off path with")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"card": card()}
    parts = a.part.split(",")
    if "c5" in parts:
        bench_c5(out, a.reps)
    if "kernel" in parts:
        bench_kernel(out)
    if "batch" in parts:
        bench_batch(out, a.reps)
    if a.ab:
        bench_ab(out, pathlib.Path(a.ab).resolve(), 10)
    out["card_after"] = card()
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        pathlib.Path(a.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
