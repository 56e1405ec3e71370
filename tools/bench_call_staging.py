"""Per-call wall time of the entry points that stage their arrays through the call buffer, two builds of libsvi_gpu.so A/B.

  python tools/bench_call_staging.py --out DIR [--lib-a PATH] [--lib-b PATH] [--rounds 4] [--calls 200]

Each round runs one worker process per build (SVI_GPU_LIB selects the build), the two alternating and swapping who goes first.
A worker times --calls synchronous calls of each entry point (after 20 warm-up calls) on one context and reports the medians:
describe and triangulate_right / triangulate_left at n = 1 and n = 1000, track_landmarks on a C3 landmark state (all stages),
stereo_frame_masked with the state's landmark centres, optimize_landmarks (1000 landmarks, 6 measurements each),
solve_stereo_posit (1000 measurements) and track_frame_stereo_only on the same state.  The inputs are seeded and shared by both
builds; every worker's outputs are hashed, and the hashes of A and B must agree.  The run-to-run spread of a build is the range
of its round medians over their median.  Writes DIR/call_staging.json (and prints a summary), with the card's name and power
limit read in the same run."""
from __future__ import annotations

import argparse
import hashlib
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


def _cams():
    from svi_mapper_b200 import load_camera
    return load_camera(str(CALIB / "vi_sensor_left.txt")), load_camera(str(CALIB / "vi_sensor_right.txt"))


def make_inputs(path: pathlib.Path):
    """The C3 frame and landmark state (SequenceTracker before frame 8 of the vi_sensor sequence, true poses) and the seeded
    query arrays, saved for the workers."""
    from svi_mapper_b200 import StereoFrontend
    from svi_mapper_b200.sequence import GpuBackend, SequenceTracker, render_sequence
    from test_call_buffer import _optimize_args, _posit_args
    cams = _cams()
    L, R, T = render_sequence(cams[0], cams[1], 9, 4000)
    with StereoFrontend(*cams, max_corners=4000) as fe:
        trk = SequenceTracker(GpuBackend(fe), cams[0])
        for t in range(8):
            trk.process(L[t], R[t], T[t])
        st = {k: v.copy() for k, v in trk.s.items()}
    rng = np.random.default_rng(3)
    W, H = cams[0].width, cams[0].height
    xy = np.stack([rng.integers(28, W - 28, 1000), rng.integers(28, H - 28, 1000)], 1).astype(np.float32)
    opt = _optimize_args(cams, 1000, 6, rng)
    posit = _posit_args(cams, 1000, rng)
    d = dict(L=L[8], R=R[8], T=T[8], T_prev=T[7], xy=xy, desc=rng.integers(0, 256, (1000, 32), dtype=np.uint8),
             search=rng.uniform(0.5, 90.0, 1000).astype(np.float32), **{"st_" + k: v for k, v in st.items()},
             **{f"opt_{i}": v for i, v in enumerate(opt)}, **{f"posit_{i}": v for i, v in enumerate(posit)})
    np.savez(path, **d)
    return len(st["uid"])


def worker(inputs: str, calls: int):
    from svi_mapper_b200 import StereoFrontend
    from test_call_buffer import _flat
    d = dict(np.load(inputs))
    st = {k[3:]: v for k, v in d.items() if k.startswith("st_")}
    n_lm = len(st["uid"])
    L, R, T, T_prev, xy, desc, search = (d[k] for k in ("L", "R", "T", "T_prev", "xy", "desc", "search"))
    opt = [d[f"opt_{i}"] for i in range(7)]
    posit = [d[f"posit_{i}"] for i in range(4)]
    tl_r = np.stack([np.maximum(0, xy[:, 0] - 28 - search), xy[:, 1] - 28], 1).astype(np.float32)
    tl_l = np.stack([xy[:, 0] - 28, xy[:, 1] - 28], 1).astype(np.float32)
    centres = np.ascontiguousarray(st["uv_ref"].astype(np.float32))
    with StereoFrontend(*_cams()) as fe:
        entries = {}
        for n in (1, 1000):
            entries[f"describe n={n}"] = lambda n=n: fe.describe(L, xy[:n])
            entries[f"triangulate_right n={n}"] = lambda n=n: fe.triangulate_right(R, tl_r[:n], xy[:n], desc[:n])
            entries[f"triangulate_left n={n}"] = lambda n=n: fe.triangulate_left(L, search[:n], tl_l[:n], xy[:n], desc[:n])
        entries[f"track_landmarks n={n_lm}"] = lambda: fe.track_landmarks(
            L, R, T, st["xyz_w"], st["last_desc_l"], st["last_desc_r"], st["last_disp"], 7.0, 1.2, uv_reference_left=st["uv_ref"],
            desc_reference_left=st["ref_desc_l"], T_left_to_world_at_detection=st["T_det"])
        entries[f"stereo_frame_masked centres={n_lm}"] = lambda: fe.add_new_landmarks(L, R, mask_centres=centres)
        entries["optimize_landmarks n=1000 m=6000"] = lambda: fe.optimize_landmarks(*opt)
        entries["solve_stereo_posit n=1000"] = lambda: fe.solve_stereo_posit(*posit)
        entries[f"track_frame_stereo_only n={n_lm}"] = lambda: fe.track_frame_stereo_only(
            L, R, st["xyz_w"], st["last_desc_l"], st["last_desc_r"], st["last_disp"], 7.0, st["uv_ref"], st["ref_desc_l"], st["T_det"],
            np.ones(n_lm, np.uint8), T, T_prev, T_prev, np.zeros(3), 1.2)
        res = {}
        for name, f in entries.items():
            for _ in range(20):
                out = f()
            h = hashlib.sha256()
            for b in _flat(out):
                h.update(b)
            ts = []
            for _ in range(calls):
                t0 = time.perf_counter()
                f()
                ts.append(time.perf_counter() - t0)
            res[name] = dict(median_us=1e6 * float(np.median(ts)), sha256=h.hexdigest())
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--lib-a", default=str(ROOT / "svi_mapper_b200" / "libsvi_gpu.so"))
    ap.add_argument("--lib-b", default=None)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        return worker(a.worker, a.calls)
    import bench_posit as bp
    out = pathlib.Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    tmp = pathlib.Path(tempfile.mkdtemp())
    n_lm = make_inputs(tmp / "inputs.npz")
    libs = {"A": a.lib_a, "B": a.lib_b or a.lib_a}
    runs = {k: [] for k in libs}
    for r in range(a.rounds):
        for k in (("A", "B") if r % 2 == 0 else ("B", "A")):
            p = subprocess.run([sys.executable, __file__, "--worker", str(tmp / "inputs.npz"), "--calls", str(a.calls)],
                               env=dict(os.environ, SVI_GPU_LIB=libs[k]), capture_output=True, text=True)
            if p.returncode != 0:
                raise RuntimeError(p.stderr)
            runs[k].append(json.loads(p.stdout.strip().splitlines()[-1]))
    rec = dict(card=bp.card(), libs=libs, rounds=a.rounds, calls=a.calls, landmarks=n_lm, entries={})
    for name in runs["A"][0]:
        e = {}
        for k in libs:
            med = [run[name]["median_us"] for run in runs[k]]
            e[k] = dict(round_medians_us=med, median_us=float(np.median(med)), spread=float((max(med) - min(med)) / np.median(med)))
        hashes = {run[name]["sha256"] for k in libs for run in runs[k]}
        e["same_outputs"] = len(hashes) == 1
        e["b_over_a"] = e["B"]["median_us"] / e["A"]["median_us"]
        rec["entries"][name] = e
    (out / "call_staging.json").write_text(json.dumps(rec, indent=1) + "\n")
    print(rec["card"])
    for name, e in rec["entries"].items():
        print(f"{name:40s} A {e['A']['median_us']:9.1f} us (spread {100 * e['A']['spread']:4.1f} %)  B {e['B']['median_us']:9.1f} us "
              f"(spread {100 * e['B']['spread']:4.1f} %)  B/A {e['b_over_a']:.3f}  same outputs {e['same_outputs']}")


if __name__ == "__main__":
    main()
