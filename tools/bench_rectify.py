"""Cost of rectifying raw images on the GPU (svi_set_rectification), one JSON line on stdout.

  batch     frames/s of svi_stereo_frames_device over --frames vi_sensor 752 x 480 pairs resident on the device (4096 pairs =
            2.9 GB of raw input, far more than the L2), once on the raw frames with rectification set and once on the same
            frames rectified by cv2.remap without it; the two arms alternate, and their outputs are compared byte for byte
  latency   time per svi_stereo_frame_masked call (one pair, ~60 landmark centres), with and without
  c3        ms per frame of the 60-frame C3 sequence rendered raw and tracked with rectification on (and the cv2-rectified
            sequence without it), SequenceTracker + GpuBackend
  kernel    rectify_kernel time per pair from torch.profiler (CUDA activities, a run of its own) over the batch arm, and the
            achieved bytes/s against the counted bytes: 2*W*H read + 2*W*H written + the two maps (6 B per pixel each) once
            per chunk
  cpu       cv2.remap per pair on one host thread with setUseOptimized(False), as the reference runs it

python tools/bench_rectify.py [--frames 4096] [--steps 5] [--out FILE]"""
from __future__ import annotations

import argparse
import json
import pathlib
import subprocess
import sys
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")[:2]
    return dict(gpu=name, power_limit=power)


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--c3-frames", type=int, default=60)
    ap.add_argument("--out")
    a = ap.parse_args(argv)
    import cv2
    import torch
    from svi_mapper_b200 import StereoFrames, StereoFrontend, _lib, load_camera
    from svi_mapper_b200.sequence import GpuBackend, SequenceTracker, render_sequence
    from svi_mapper_b200.synth import stereo_frames_range_torch, unrectify

    if not torch.cuda.is_available():
        raise SystemExit("bench_rectify: no CUDA device")
    calib = ROOT / "tests" / "golden" / "calib"
    cams = load_camera(str(calib / "vi_sensor_left.txt")), load_camera(str(calib / "vi_sensor_right.txt"))
    W, H, F = cams[0].width, cams[0].height, a.frames
    res = dict(gpu_info(), width=W, height=H, frames=F)
    cv2.setUseOptimized(False)
    maps = [cv2.initUndistortRectifyMap(c.K, c.distortion, c.rectification, c.P, (W, H), cv2.CV_16SC2) for c in cams]

    # ---- CPU reference: cv2.remap of both images of a pair on one thread
    cv2.setNumThreads(1)
    rl, rr = stereo_frames_range_torch(0, 8, W, H, 7)
    rl, rr = rl.cpu().numpy(), rr.cpu().numpy()
    t0 = time.perf_counter()
    for i in range(8):
        cv2.remap(rl[i], *maps[0], cv2.INTER_LINEAR)
        cv2.remap(rr[i], *maps[1], cv2.INTER_LINEAR)
    res["cpu_remap_ms_per_pair"] = round(1e3 * (time.perf_counter() - t0) / 8, 4)
    cv2.setNumThreads(-1)

    # ---- batch, device-resident
    raw_l, raw_r = stereo_frames_range_torch(0, F, W, H, 11)
    rect_l = torch.empty_like(raw_l)
    rect_r = torch.empty_like(raw_r)
    for f0 in range(0, F, 256):                       # cv2.remap on the host, the result back to the device
        hl, hr = raw_l[f0:f0 + 256].cpu().numpy(), raw_r[f0:f0 + 256].cpu().numpy()
        rect_l[f0:f0 + 256] = torch.from_numpy(np.stack([cv2.remap(x, *maps[0], cv2.INTER_LINEAR) for x in hl])).cuda()
        rect_r[f0:f0 + 256] = torch.from_numpy(np.stack([cv2.remap(x, *maps[1], cv2.INTER_LINEAR) for x in hr])).cuda()
    fe_raw, fe_plain = StereoFrontend(*cams), StereoFrontend(*cams)
    fe_raw.set_rectification(*cams)
    cap = fe_raw.max_corners

    def outputs():
        return dict(n_keypoints=torch.zeros(F, dtype=torch.int32, device="cuda"), n_detected=torch.zeros(F, dtype=torch.int32, device="cuda"),
                    uv_left=torch.zeros((F, cap, 2), device="cuda"), uv_right=torch.zeros((F, cap, 2), device="cuda"),
                    xyz_left=torch.zeros((F, cap, 3), dtype=torch.float64, device="cuda"), desc_left=torch.zeros((F, cap, 32), dtype=torch.uint8, device="cuda"),
                    desc_right=torch.zeros((F, cap, 32), dtype=torch.uint8, device="cuda"), distance=torch.zeros((F, cap), dtype=torch.int32, device="cuda"),
                    match_index=torch.zeros((F, cap), dtype=torch.int32, device="cuda"), status=torch.zeros((F, cap), dtype=torch.uint8, device="cuda"))
    keys = ("n_keypoints", "n_detected", "uv_left", "uv_right", "xyz_left", "desc_left", "desc_right", "distance", "match_index", "status")
    arms = {"with": (fe_raw, raw_l, raw_r, outputs()), "without": (fe_plain, rect_l, rect_r, outputs())}

    def step(arm):
        fe, l, r, o = arms[arm]
        res_ = _lib.StereoResult(cap, *(o[k].data_ptr() for k in keys))
        fe.stereo_frames_device(l.data_ptr(), r.data_ptr(), W, W * H, F, res_, None, torch.cuda.current_stream().cuda_stream)

    for arm in arms:                                   # warm-up
        step(arm)
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(a.steps):
        for arm in arms:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step(arm)
            e1.record()
            torch.cuda.synchronize()
            times[arm].append(e0.elapsed_time(e1))
    for fe, *_ in arms.values():
        fe.check_overflow()
    got = {arm: StereoFrames(**{k: v.cpu().numpy() for k, v in o.items()}) for arm, (_, _, _, o) in arms.items()}
    same = bool(np.array_equal(got["with"].n_keypoints, got["without"].n_keypoints))
    for f in range(F) if same else ():
        x, y = got["with"].frame(f), got["without"].frame(f)
        if not all(x[k].tobytes() == y[k].tobytes() for k in x):
            same = False
            break
    fps = {arm: F / (np.median(t) / 1e3) for arm, t in times.items()}
    res["batch"] = dict(frames_per_s_with=round(fps["with"]), frames_per_s_without=round(fps["without"]),
                        ms_per_step_with=[round(t, 3) for t in times["with"]], ms_per_step_without=[round(t, 3) for t in times["without"]],
                        loss_percent=round(100.0 * (1.0 - fps["with"] / fps["without"]), 2), outputs_identical=same,
                        kernels_per_chunk_with=fe_raw.kernels_per_chunk(F), kernels_per_chunk_without=fe_plain.kernels_per_chunk(F))

    # ---- rectify_kernel on its own (profiler run of its own, after the timed steps)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step("with")
        torch.cuda.synchronize()
    ev = [e for e in prof.key_averages() if "rectify_kernel" in e.key]
    k_us = sum(getattr(e, "device_time_total", 0.0) or getattr(e, "cuda_time_total", 0.0) for e in ev)
    chunk = fe_raw.config()["chunk_frames"]
    n_pad = (W * H + 7) // 8 * 8
    bytes_pair = 2 * W * H + 2 * W * H + 2 * 6 * n_pad / chunk
    res["kernel"] = dict(launches=sum(e.count for e in ev), us_per_pair=round(k_us / F, 4), counted_bytes_per_pair=round(bytes_pair),
                         achieved_GB_per_s=round(bytes_pair * F / (k_us * 1e-6) / 1e9, 1) if k_us else None, chunk_frames=chunk)
    del arms, got, raw_l, raw_r, rect_l, rect_r
    torch.cuda.empty_cache()

    # ---- latency: one pair per call
    L, R = stereo_frames_range_torch(0, 2, W, H, 3)
    L, R = L.cpu().numpy(), R.cpu().numpy()
    Lr, Rr = cv2.remap(L[0], *maps[0], cv2.INTER_LINEAR), cv2.remap(R[0], *maps[1], cv2.INTER_LINEAR)
    centres = np.random.default_rng(1).uniform([0, 0], [W, H], (60, 2)).astype(np.float32)
    lat = {}
    for arm, fe, x, y in (("with", fe_raw, L[0], R[0]), ("without", fe_plain, Lr, Rr)):
        for _ in range(20):
            fe.add_new_landmarks(x, y, mask_centres=centres)
        t0 = time.perf_counter()
        for _ in range(300):
            fe.add_new_landmarks(x, y, mask_centres=centres)
        lat[arm] = (time.perf_counter() - t0) / 300 * 1e3
    res["latency_ms_per_call"] = {"with": round(lat["with"], 4), "without": round(lat["without"], 4)}

    # ---- C3: the raw sequence tracked with rectification on
    n = a.c3_frames
    Ls, Rs, T = render_sequence(cams[0], cams[1], n, 4000)
    RLs, RRs = np.stack([unrectify(x, cams[0]) for x in Ls]), np.stack([unrectify(x, cams[1]) for x in Rs])
    CLs = np.stack([cv2.remap(x, *maps[0], cv2.INTER_LINEAR) for x in RLs])
    CRs = np.stack([cv2.remap(x, *maps[1], cv2.INTER_LINEAR) for x in RRs])
    c3 = {}
    logs = {}
    for arm, fe, A, B in (("with", fe_raw, RLs, RRs), ("without", fe_plain, CLs, CRs)):
        tr = SequenceTracker(GpuBackend(fe), cams[0])
        ms = []
        for t in range(n):
            t0 = time.perf_counter()
            tr.process(A[t], B[t], T[t])
            ms.append((time.perf_counter() - t0) * 1e3)
        c3[arm] = float(np.mean(ms[3:]))
        logs[arm] = tr.log
    res["c3_ms_per_frame"] = dict(with_rectification=round(c3["with"], 4), without=round(c3["without"], 4),
                                  logs_identical=logs["with"] == logs["without"], frames=n)
    fe_raw.close()
    fe_plain.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
