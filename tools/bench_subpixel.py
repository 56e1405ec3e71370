#!/usr/bin/env python3
"""Sub-pixel disparity (svi_params.subpixel_window / subpixel_search) on a B200: what the refinement costs.  Prints one
JSON object (--out: also writes it there).  Every leg first compares the outputs of the mode on with the CPU
restatement's refinement (tests/subpixel_np.py) of the mode-off outputs, bit for bit, then times.

  batch    C2-shaped device-resident batch (4096 x 1241 x 376, maxCorners 2000): frames/s of svi_stereo_frames_device
           with the mode off and on (w = L = 5), CUDA events around `reps` calls, the two alternated twice in one process
  kernel   torch.profiler (a separate run): subpixel_refine_kernel's device time per 64-frame chunk of that batch
  masked   svi_stereo_frame_masked on one vi_sensor pair with 300 landmark centres: median latency off / on, alternated
  c5       the C5 sparse frame (3840 x 1080, maxCorners 10000, +-1 row band): median latency off / on, alternated
The card's name, power limit and SM clock are read in the same run."""
import argparse
import json
import pathlib
import sys
import time
from types import SimpleNamespace

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))

from bench_c5 import BANDS, H5, K5, RANGE5, W5, card, kitti  # noqa: E402
import subpixel_np as sp  # noqa: E402
from oracle import frontend_np as o  # noqa: E402
from svi_mapper_b200 import StereoFrontend, _lib, load_camera  # noqa: E402
from svi_mapper_b200.synth import stereo_pair  # noqa: E402

WL = dict(subpixel_window=5, subpixel_search=5)
C2 = dict(max_corners=2000)


def tri_of(cams):
    cl, cr = cams
    return o.Triangulator(o.Camera(cl.width, cl.height, np.asarray(cl.P, np.float64).reshape(3, 4)),
                          o.Camera(cr.width, cr.height, np.asarray(cr.P, np.float64).reshape(3, 4)))


def check(on: dict, off: dict, L, R, tri, what):
    """on == the restatement's refinement of off (status, uv_right, xyz_left), the rest unchanged; returns the slot counts."""
    for k in ("uv_l", "desc_l", "dist", "idx"):
        assert np.array_equal(on[k], off[k]), (what, k)
    uv_r, xyz, st = sp.subpixel_refine(L, R, off["uv_l"], off["uv_r"], off["status"], 5, 5, tri)
    ok = st == o.ST_OK
    assert np.array_equal(on["status"], st), (what, "status")
    assert np.array_equal(on["uv_r"][ok], uv_r[ok]) and np.array_equal(on["xyz"][ok], xyz[ok]), (what, "uv_r / xyz")
    return dict(ok_off=int((off["status"] == o.ST_OK).sum()), ok_on=int(ok.sum()), rejected=int((st == sp.ST_SUBPIXEL_REJECTED).sum()))


def c2_inputs(n):
    import torch
    cams = kitti()
    W, H = cams[0].width, cams[0].height
    base = [stereo_pair(W, H, s) for s in range(1000, 1016)]
    Ls = torch.from_numpy(np.stack([base[i % 16][0] for i in range(n)])).cuda()
    Rs = torch.from_numpy(np.stack([base[i % 16][1] for i in range(n)])).cuda()
    return cams, base, Ls, Rs


def device_result(fe, n):
    import torch
    from svi_mapper_b200.frontend import StereoFrames
    host = StereoFrames.empty(1, 1)
    dev = {k: torch.zeros((n,) if v.ndim == 1 else (n, fe.max_corners) + v.shape[2:], dtype=torch.from_numpy(v).dtype, device="cuda")
           for k, v in vars(host).items() if v is not None}
    r = _lib.StereoResult(fe.max_corners, *[dev[k].data_ptr() for k in ("n_keypoints", "n_detected", "uv_left", "uv_right", "xyz_left",
                                                                         "desc_left", "desc_right", "distance", "match_index", "status")])
    return dev, r


def bench_batch(out, reps, n=4096):
    import torch
    from svi_mapper_b200.frontend import StereoFrames
    cams, base, Ls, Rs = c2_inputs(n)
    W, H = cams[0].width, cams[0].height
    tri = tri_of(cams)
    stream = torch.cuda.current_stream().cuda_stream
    with StereoFrontend(*cams, **C2) as off, StereoFrontend(*cams, **C2, **WL) as on:
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
            counts.append(check(fr["on"], fr["off"], base[f % 16][0], base[f % 16][1], tri, f"batch frame {f}"))
        for k in ("n_keypoints", "n_detected", "distance", "match_index", "uv_left"):
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
    with StereoFrontend(*cams, **C2, **WL) as fe:
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
        sub = [v for k, v in per.items() if "subpixel_refine_kernel" in k]
        out["kernel_c2"] = dict(chunk_frames=chunk, chunks=chunks, subpixel_refine_kernel=sub[0] if sub else None,
                                all_kernels_us_per_chunk=float(sum(v["us_per_chunk"] for v in per.values())), per_kernel=per)


def median_ms(fns, reps):
    """Medians of synchronous calls, the callables alternated."""
    t = {k: [] for k in fns}
    for k, f in list(fns.items()) * 3:
        f()
    for _ in range(reps):
        for k, f in fns.items():
            t0 = time.perf_counter()
            f()
            t[k].append(time.perf_counter() - t0)
    return {k: float(np.median(v) * 1e3) for k, v in t.items()}


def bench_masked(out, reps):
    calib = ROOT / "tests" / "golden" / "calib"
    cams = load_camera(str(calib / "vi_sensor_left.txt")), load_camera(str(calib / "vi_sensor_right.txt"))
    W, H = cams[0].width, cams[0].height
    L, R = stereo_pair(W, H, 4000)
    centres = np.random.default_rng(1).uniform([0, 0], [W, H], (300, 2)).astype(np.float32)
    with StereoFrontend(*cams) as off, StereoFrontend(*cams, **WL) as on:
        c = check(on.add_new_landmarks(L, R, mask_centres=centres), off.add_new_landmarks(L, R, mask_centres=centres), L, R, tri_of(cams),
                  "masked")
        ms = median_ms({k: (lambda fe=fe: fe.add_new_landmarks(L, R, mask_centres=centres)) for k, fe in (("off", off), ("on", on))}, reps)
    out["masked_vi_sensor"] = dict(outputs_checked=c, reps=reps, median_ms=ms)


def bench_c5(out, reps):
    k0, k1 = kitti()
    cams = SimpleNamespace(width=W5, height=H5, P=k0.P), SimpleNamespace(width=W5, height=H5, P=k1.P)
    L, R = stereo_pair(W5, H5, 3000, d_max=900)
    kw = dict(max_corners=K5, search_range_px=RANGE5, max_candidates=131072, chunk_frames=1)
    band = BANDS["band_pm1"]
    with StereoFrontend(*cams, **kw) as off, StereoFrontend(*cams, **kw, **WL) as on:
        c = check(on.stereo_frames_sparse(L, R, None, *band).frame(0), off.stereo_frames_sparse(L, R, None, *band).frame(0), L, R,
                  tri_of(cams), "c5 sparse")
        ms = median_ms({k: (lambda fe=fe: fe.stereo_frames_sparse(L, R, None, *band)) for k, fe in (("off", off), ("on", on))}, reps)
    out["c5_sparse"] = dict(band=band, outputs_checked=c, reps=reps, median_ms=ms)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--part", default="batch,kernel,masked,c5", help="comma list of batch, kernel, masked, c5")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"card": card(), "subpixel": WL}
    parts = a.part.split(",")
    if "batch" in parts:
        bench_batch(out, a.reps)
    if "kernel" in parts:
        bench_kernel(out)
    if "masked" in parts:
        bench_masked(out, 20 * a.reps)
    if "c5" in parts:
        bench_c5(out, a.reps)
    out["card_after"] = card()
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(a.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
