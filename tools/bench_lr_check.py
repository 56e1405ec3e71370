#!/usr/bin/env python3
"""Dense left-right check (svi_params.lr_max_diff) on a B200: what the check costs.  Prints one JSON object (--out: also
writes it there).  Every leg first compares the outputs of the check on with the CPU restatement's check
(tests/lr_check_np.py) of the check-off outputs, byte for byte, then times.

  batch    C2-shaped device-resident batch (4096 x 1241 x 376, maxCorners 2000): frames/s of svi_stereo_frames_device with
           the check off and on (lr_max_diff = 1), CUDA events around `reps` calls, the two alternated twice in one process
  kernel   torch.profiler (a separate run): lr_check_kernel's device time per 64-frame chunk of that batch, next to the
           forward matcher's (stereo_match_binned_kernel on C2)
  masked   svi_stereo_frame_masked on one vi_sensor pair with 300 landmark centres: median latency off / on, alternated
The card's name, power limit and SM clock are read in the same run."""
import argparse
import json
import pathlib
import sys

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))

from bench_c5 import card  # noqa: E402
from bench_subpixel import C2, c2_inputs, device_result, median_ms, tri_of  # noqa: E402
import lr_check_np as lr  # noqa: E402
from oracle import frontend_np as o  # noqa: E402
from svi_mapper_b200 import StereoFrontend, load_camera  # noqa: E402
from svi_mapper_b200.synth import stereo_pair  # noqa: E402

LR = dict(lr_max_diff=1)


def check(on: dict, off: dict, L, tri, what):
    """on == off with the restatement's check applied to its status, every other field unchanged; returns the slot counts."""
    for k in ("uv_l", "desc_l", "dist", "idx"):
        assert np.array_equal(on[k], off[k]), (what, k)
    ok = off["status"] == o.ST_OK
    for k in ("uv_r", "xyz", "desc_r"):
        assert np.array_equal(on[k][ok], off[k][ok]), (what, k)
    st = lr.lr_check(L, off["uv_l"], off["uv_r"], off["desc_r"], off["status"], LR["lr_max_diff"], tri)
    assert np.array_equal(on["status"], st), (what, "status")
    return dict(ok_off=int(ok.sum()), ok_on=int((st == o.ST_OK).sum()), rejected=int((st == lr.ST_LR_INCONSISTENT).sum()))


def bench_batch(out, reps, n=4096):
    import torch
    from svi_mapper_b200.frontend import StereoFrames
    cams, base, Ls, Rs = c2_inputs(n)
    W, H = cams[0].width, cams[0].height
    tri = tri_of(cams)
    stream = torch.cuda.current_stream().cuda_stream
    with StereoFrontend(*cams, **C2) as off, StereoFrontend(*cams, **C2, **LR) as on:
        fes = {"off": off, "on": on}
        res = {k: device_result(fe, n) for k, fe in fes.items()}

        def call(k):
            fes[k].stereo_frames_device(Ls.data_ptr(), Rs.data_ptr(), W, W * H, n, res[k][1], stream=stream)
        for k in ("off", "on"):
            call(k)
        torch.cuda.synchronize()
        counts = []
        for f in (0, 1, n - 1):   # outputs first
            fr = {k: StereoFrames(**{q: v[f:f + 1].cpu().numpy() for q, v in res[k][0].items()}).frame(0) for k in fes}
            counts.append(check(fr["on"], fr["off"], base[f % 16][0], tri, f"batch frame {f}"))
        for k in ("n_keypoints", "n_detected", "distance", "match_index", "uv_left", "desc_left"):
            assert torch.equal(res["on"][0][k], res["off"][0][k]), k
        t = {"off": [], "on": []}
        for k in ("off", "on", "off", "on"):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                call(k)
            e1.record()
            torch.cuda.synchronize()
            fes[k].check_overflow()
            t[k].append(n / (e0.elapsed_time(e1) / reps) * 1e3)
        out["batch_c2_x4096"] = dict(frames=n, reps=reps, outputs_checked=counts, kernels_per_chunk={k: fe.kernels_per_chunk(n) for k, fe in fes.items()},
                                     chunk_frames={k: fe.config()["chunk_frames"] for k, fe in fes.items()},
                                     frames_per_s={k: v for k, v in t.items()},
                                     mean_frames_per_s={k: float(np.mean(v)) for k, v in t.items()},
                                     cost_pct=float(100.0 * (1.0 - np.mean(t["on"]) / np.mean(t["off"]))))


def bench_kernel(out, n=4096):
    import torch
    from torch.profiler import ProfilerActivity, profile
    cams, _, Ls, Rs = c2_inputs(n)
    W, H = cams[0].width, cams[0].height
    with StereoFrontend(*cams, **C2, **LR) as fe:
        _, r = device_result(fe, n)
        chunk = fe.config()["chunk_frames"]
        fe.stereo_frames_device(Ls.data_ptr(), Rs.data_ptr(), W, W * H, n, r)
        torch.cuda.synchronize()
        reps = 3
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                fe.stereo_frames_device(Ls.data_ptr(), Rs.data_ptr(), W, W * H, n, r)
            torch.cuda.synchronize()
        chunks = reps * ((n + chunk - 1) // chunk)
        per = {e.key: dict(us_per_chunk=e.device_time_total / chunks, launches=e.count) for e in prof.key_averages() if e.device_time_total > 0}

        def find(name):
            hit = [v for k, v in per.items() if name in k]
            return hit[0] if hit else None
        out["kernel_c2"] = dict(chunk_frames=chunk, chunks=chunks, lr_check_kernel=find("lr_check_kernel"),
                                stereo_match_binned_kernel=find("stereo_match_binned_kernel"),
                                all_kernels_us_per_chunk=float(sum(v["us_per_chunk"] for v in per.values())), per_kernel=per)


def bench_masked(out, reps):
    calib = ROOT / "tests" / "golden" / "calib"
    cams = load_camera(str(calib / "vi_sensor_left.txt")), load_camera(str(calib / "vi_sensor_right.txt"))
    W, H = cams[0].width, cams[0].height
    L, R = stereo_pair(W, H, 4000)
    centres = np.random.default_rng(1).uniform([0, 0], [W, H], (300, 2)).astype(np.float32)
    with StereoFrontend(*cams) as off, StereoFrontend(*cams, **LR) as on:
        c = check(on.add_new_landmarks(L, R, mask_centres=centres), off.add_new_landmarks(L, R, mask_centres=centres), L, tri_of(cams),
                  "masked")
        ms = median_ms({k: (lambda fe=fe: fe.add_new_landmarks(L, R, mask_centres=centres)) for k, fe in (("off", off), ("on", on))}, reps)
    out["masked_vi_sensor"] = dict(outputs_checked=c, reps=reps, median_ms=ms)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--part", default="batch,kernel,masked", help="comma list of batch, kernel, masked")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"card": card(), "lr_check": LR}
    parts = a.part.split(",")
    if "batch" in parts:
        bench_batch(out, a.reps)
    if "kernel" in parts:
        bench_kernel(out)
    if "masked" in parts:
        bench_masked(out, 20 * a.reps)
    out["card_after"] = card()
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(a.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
