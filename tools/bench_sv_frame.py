"""Cost of one stereo-only tracking frame as one call (svi_track_frame_stereo_only) against the composed calls it replaces.

  python tools/bench_sv_frame.py --out DIR [--reps 30] [--frames 60]

1. Python, on the same C3 landmark states (the SequenceTracker's state before frames 8 .. 19 of the vi_sensor sequence, true-pose
   priors, every landmark a pose candidate): median wall time of the fused call and of the composed calls (track_landmarks
   stages 1-2, solve_stereo_posit, track_landmarks stage 3, stage 2 on the regional set, with the numpy routing in between),
   --reps alternating repetitions per state; the outputs of the two are compared.
2. The C++ tracker CTrackerSV over --frames C3 frames (facade_demo --sequence-sv, SVI_DEMO_TIMING): the fused frame call (default)
   against the composed calls with the CPU solve (SVI_HOST_POSIT=cpu), two alternating runs each.
3. tools/bench_posit.py in the same run (the solve alone, and the sequence split).
Writes DIR/r3_sv_frame.json (and prints it), with the card's name and power limit read in the same run."""
from __future__ import annotations

import argparse
import json
import pathlib
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))
sys.dont_write_bytecode = True

CALIB = ROOT / "tests" / "golden" / "calib"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--frames", type=int, default=60)
    a = ap.parse_args()
    import bench_posit as bp
    import test_sv_frame as tsf
    from svi_mapper_b200 import StereoFrontend
    from svi_mapper_b200.sequence import GpuBackend, SequenceTracker, render_sequence
    out = pathlib.Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    cams = tsf._cams()
    rec = dict(card=bp.card(), reps=a.reps, python=[], sequence={})
    L, R, T = render_sequence(cams[0], cams[1], max(a.frames, 20), 4000)
    with StereoFrontend(*cams, max_corners=4000) as fe:
        trk = SequenceTracker(GpuBackend(fe), cams[0])
        for k in range(20):
            if k >= 8:
                st = {kk: v.copy() for kk, v in trk.s.items()}
                args = (L[k], R[k], st, np.ones(len(st["uid"]), np.uint8), T[k], T[k - 1], T[k - 1], np.zeros(3), 1.2)
                for _ in range(3):
                    want, got = tsf.composed(fe, *args), tsf.fused(fe, *args)
                tsf.assert_same(got, want, f"frame {k}")
                tf, tc = [], []
                for _ in range(a.reps):
                    t0 = time.perf_counter()
                    tsf.fused(fe, *args)
                    t1 = time.perf_counter()
                    tsf.composed(fe, *args)
                    t2 = time.perf_counter()
                    tf.append(t1 - t0)
                    tc.append(t2 - t1)
                row = dict(frame=k, landmarks=len(st["uid"]), pose_hits=int((got["pose_stage"]["stage"] > 0).sum()),
                           epipolar=int((got["route"] == 2).sum()), regional=int(((got["route"] == 3) | (got["route"] == 4)).sum()),
                           source=got["source"], fused_median_ms=1e3 * float(np.median(tf)), composed_median_ms=1e3 * float(np.median(tc)))
                print(row, flush=True)
                rec["python"].append(row)
            trk.process(L[k], R[k], T[k])
    rec["python_median_fused_ms"] = float(np.median([r["fused_median_ms"] for r in rec["python"]]))
    rec["python_median_composed_ms"] = float(np.median([r["composed_median_ms"] for r in rec["python"]]))
    tmp = pathlib.Path(tempfile.mkdtemp())
    n = a.frames
    L[:n].tofile(tmp / "L.raw")
    R[:n].tofile(tmp / "R.raw")
    argv = ["--sequence-sv", str(CALIB / "vi_sensor_left.txt"), str(CALIB / "vi_sensor_right.txt"), str(n), str(tmp / "L.raw"), str(tmp / "R.raw"), "4000"]
    for mode in ("gpu", "cpu", "gpu", "cpu"):
        rec["sequence"].setdefault("fused" if mode == "gpu" else "composed_cpu_solve", []).append(json.loads(bp.demo(argv + [str(tmp / "unused.txt")], mode, 1)[0]))
    r = subprocess.run([sys.executable, str(ROOT / "tools" / "bench_posit.py"), "--out", str(tmp), "--calls", "100"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(r.stderr)
    rec["bench_posit"] = json.loads((tmp / "r3_posit.json").read_text())
    (out / "r3_sv_frame.json").write_text(json.dumps(rec, indent=1) + "\n")
    print(json.dumps({k: v for k, v in rec.items() if k not in ("python", "bench_posit")}))
    print(json.dumps({k: v for k, v in rec["bench_posit"].items() if k != "sequence"}))


if __name__ == "__main__":
    main()
