"""Cost of the pose solve of the stereo-only tracker on the GPU (svi_solve_stereo_posit) against the C++ host's CPU loop.

  python tools/bench_posit.py --out DIR [--calls 200] [--frames 60]

1. The solve alone, on the same seeded vi_sensor problems at 100 / 500 / 1000 / 2000 / 4000 measurements (prior 2 cm / 1 deg
   off, 10 % outliers): median wall time of one synchronous call over --calls calls, through the Python binding and through
   the C++ host layer (facade_demo --posit: GPU call, and the CPU loop under SVI_HOST_POSIT=cpu); the outputs are compared.
2. The C3 sequence (render_sequence, vi_sensor, --frames frames) through CTrackerSV (facade_demo --sequence-sv): median frame
   time and the split pose stage / solves / trackEpipolar / optimisation / re-detection, with the GPU solve and with the CPU
   loop, two alternating runs each; plus the pose error against the ground truth.
Writes DIR/r3_posit.json (and prints it), with the card's name and power limit read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.dont_write_bytecode = True

CALIB = ROOT / "tests" / "golden" / "calib"
EXE = ROOT / "svi_mapper_b200" / "host" / "facade_demo"


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def demo(args, mode, timing=None):
    env = dict(os.environ)
    env.pop("SVI_HOST_POSIT", None)
    env.pop("SVI_DEMO_TIMING", None)
    if mode == "cpu":
        env["SVI_HOST_POSIT"] = "cpu"
    if timing:
        env["SVI_DEMO_TIMING"] = str(timing)
    r = subprocess.run([str(EXE), *args], capture_output=True, text=True, env=env)
    if r.returncode != 0:
        raise RuntimeError(r.stderr)
    return r.stdout.strip().splitlines()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--frames", type=int, default=60)
    a = ap.parse_args()
    import test_stereo_posit as tsp
    from svi_mapper_b200 import StereoFrontend
    from svi_mapper_b200.sequence import render_sequence
    out = pathlib.Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    cams = tsp._cams("vi_sensor")
    P_l, P_r = np.asarray(cams[0].P).reshape(3, 4), np.asarray(cams[1].P).reshape(3, 4)
    rec = dict(card=card(), calls=a.calls, solve=[], sequence={})
    tmp = pathlib.Path(tempfile.mkdtemp())
    with StereoFrontend(*cams) as fe:
        for n in (100, 500, 1000, 2000, 4000):
            rng = np.random.default_rng(100 + n)
            T_true = tsp._pose([0.2, 1.0, 0.1], 0.03, [0.06, -0.02, 0.12])
            xyz = np.c_[rng.uniform(-4, 4, n), rng.uniform(-2, 2, n), rng.uniform(3, 25, n)]
            uvl, uvr = tsp._observe(P_l, P_r, T_true, xyz, rng)
            bad = rng.random(n) < 0.1
            uvl[bad] += rng.uniform(-40, 40, (int(bad.sum()), 2)).astype(np.float32)
            T_est = tsp._pose([1, 0, 0], np.radians(1.0), [0, 0, 0]) @ T_true
            T_est[:3, 3] += [0.02, 0.0, 0.0]
            p = dict(name=f"b{n}", xyz=xyz, uvl=uvl, uvr=uvr, T_est=T_est, T_last=np.eye(4), t_imu=np.zeros(3))
            f = tmp / f"b{n}.txt"
            tsp._write_problem(f, p)
            argv = ["--posit", str(CALIB / "vi_sensor_left.txt"), str(CALIB / "vi_sensor_right.txt"), str(f)]
            g = demo(argv, "gpu", a.calls)
            c = demo(argv, "cpu", a.calls)
            for _ in range(10):
                res = fe.solve_stereo_posit(xyz, uvl, uvr, T_est, np.eye(4), np.zeros(3))
            ts = []
            for _ in range(a.calls):
                t0 = time.perf_counter()
                res = fe.solve_stereo_posit(xyz, uvl, uvr, T_est, np.eye(4), np.zeros(3))
                ts.append(time.perf_counter() - t0)
            same = g[0] == c[0] == tsp._expected_line(res, n)
            row = dict(n=n, iterations=res["iterations"], outcome=res["outcome"], outputs_equal=bool(same),
                       cpp_gpu_median_us=json.loads(g[1])["median_us"], cpp_cpu_median_us=json.loads(c[1])["median_us"],
                       python_gpu_median_us=1e6 * float(np.median(ts)))
            print(row, flush=True)
            rec["solve"].append(row)
    n = a.frames
    L, R, T = render_sequence(cams[0], cams[1], n, 4000)
    L.tofile(tmp / "L.raw")
    R.tofile(tmp / "R.raw")
    argv = ["--sequence-sv", str(CALIB / "vi_sensor_left.txt"), str(CALIB / "vi_sensor_right.txt"), str(n), str(tmp / "L.raw"), str(tmp / "R.raw"), "4000"]
    for mode in ("gpu", "cpu", "gpu", "cpu"):
        rec["sequence"].setdefault(mode, []).append(json.loads(demo(argv + [str(tmp / "unused.txt")], mode, 1)[0]))
    lines = {}
    for mode in ("gpu", "cpu"):
        demo(argv + [str(tmp / f"sv_{mode}.txt")], mode)
        lines[mode] = (tmp / f"sv_{mode}.txt").read_text()
    rec["sequence"]["outputs_identical"] = lines["gpu"] == lines["cpu"]
    frames = tsp.parse_sequence_sv(lines["gpu"])
    err = []
    for fr, Tg in zip(frames, T):
        ce, cg = -fr["T"][:3, :3].T @ fr["T"][:3, 3], -Tg[:3, :3].T @ Tg[:3, 3]
        Rr = fr["T"][:3, :3] @ Tg[:3, :3].T
        err.append(dict(source=fr["POSE"], posit=int(fr["POSIT"]), visible=int(fr["VISIBLE"]), pos_err_cm=100 * float(np.linalg.norm(ce - cg)),
                        rot_err_deg=float(np.degrees(np.arccos(np.clip((np.trace(Rr) - 1) / 2, -1, 1))))))
    rec["sequence"]["per_frame"] = err
    (out / "sv_gpu.txt").write_text(lines["gpu"])
    (out / "r3_posit.json").write_text(json.dumps(rec, indent=1) + "\n")
    print(json.dumps({k: v for k, v in rec.items() if k != "sequence"}))
    print(json.dumps({k: v for k, v in rec["sequence"].items() if k != "per_frame"}))
    for k, e in enumerate(err):
        print(k, e)


if __name__ == "__main__":
    main()
