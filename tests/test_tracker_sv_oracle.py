"""The stereo-only tracker against an independent CPU restatement.

The pose solve: oracle/svi_oracle.c svo_solve_stereo_posit, a plain-C restatement of CSolverStereoPosit::getTransformationWORLDtoLEFT
(reference src/optimization/CSolverStereoPosit.cpp:8-170), pinned to the C++ host's CPU loop to the last printed digit and to the
numpy restatement to 1e-9.  The frame: oracle/tracker_np.sv_frame (the C tracking cascade on the candidate, epipolar and regional
subsets and the C solve) against svi_track_frame_stereo_only byte for byte, at landmark counts and flag patterns that drive the
device compaction, gather, assembly, routing and scatter past their chunk boundaries.  The sequence: oracle/tracker_np.TrackerSV
(CTrackerSV::process and the CFundamentalMatcher bookkeeping it calls) in lockstep with facade_demo --sequence-sv, every printed
number of every frame."""
import os
import pathlib
import subprocess
import sys

import numpy as np
import pytest

from svi_mapper_b200 import StereoFrontend, _lib

ROOT = pathlib.Path(__file__).resolve().parents[1]
CALIB = ROOT / "tests" / "golden" / "calib"
EXE = ROOT / "svi_mapper_b200" / "host" / "facade_demo"

pytestmark = pytest.mark.usefixtures("built_library", "built_oracle")

TRACK_KEYS = ("status", "stage", "uv_l", "uv_r", "xyz", "desc_l", "desc_r")
POSIT_KEYS = ("outcome", "iterations", "inliers", "average_squared_error", "risk")


def _cams(name="vi_sensor"):
    from svi_mapper_b200 import load_camera
    return load_camera(str(CALIB / f"{name}_left.txt")), load_camera(str(CALIB / f"{name}_right.txt"))


def _cfg(cams, mc=4000):
    from oracle import c_oracle as co
    return co.make_config(cams[0], cams[1], max_corners=mc)


def _threads():
    from oracle import c_oracle as co
    return co.host_threads()


# ------------------------------------------------------------------------------------------------------------ the pose solve
def _c_line(res, n):
    """What facade_demo --posit prints for a result of the C port (the host's what() texts, std::to_string = %f)."""
    from test_stereo_posit import _expected_line
    return _expected_line(res, n)


@pytest.mark.parametrize("cam_name,seeds", [("vi_sensor", (41, 42)), ("kitti_11_12", (43, 44))])
def test_c_solve_equals_host_cpu_loop_to_the_last_digit(cam_name, seeds, tmp_path):
    """svo_solve_stereo_posit against facade_demo --posit with SVI_HOST_POSIT=cpu (the C++ host's CPU loop, no GPU) on the seeded
    problem sets of test_stereo_posit: every OK line -- the 12 pose numbers at %.17g and the iteration count -- and every FAILED text
    byte for byte; all four outcomes that a finite input reaches occur.  Then the fields the printed line does not show: a
    failed solve returns the prior, and the fields its outcome does not compute are zero."""
    from oracle import c_oracle as co
    from test_stereo_posit import _demo_posit, make_problems
    cams = _cams(cam_name)
    P_l, P_r = np.asarray(cams[0].P).reshape(3, 4), np.asarray(cams[1].P).reshape(3, 4)
    outcomes = set()
    for seed in seeds:
        for p in make_problems(cams, seed):
            res = co.solve_stereo_posit(P_l, P_r, p["xyz"], p["uvl"], p["uvr"], p["T_est"], p["T_last"], p["t_imu"])
            assert _c_line(res, len(p["xyz"])) == _demo_posit(cam_name, p, tmp_path, "cpu"), (cam_name, seed, p["name"], res)
            outcomes.add(res["outcome"])
            if res["outcome"] != _lib.SVI_POSIT_OK:
                assert res["T"].tobytes() == np.asarray(p["T_est"], np.float64).tobytes()
            if res["outcome"] == _lib.SVI_POSIT_TOO_FEW_POINTS:
                assert (res["iterations"], res["inliers"], res["average_squared_error"], res["risk"]) == (0, 0, 0.0, 0.0)
            if res["outcome"] == _lib.SVI_POSIT_INACCURATE:
                assert res["risk"] == 0.0
    assert outcomes == {_lib.SVI_POSIT_OK, _lib.SVI_POSIT_TOO_FEW_POINTS, _lib.SVI_POSIT_INACCURATE, _lib.SVI_POSIT_HIGH_RISK}, outcomes


@pytest.mark.parametrize("cam_name,seed", [("vi_sensor", 45), ("kitti_11_12", 46)])
def test_c_solve_matches_numpy_restatement(cam_name, seed):
    """The C port against oracle.frontend_np.solve_stereo_posit (vectorised sums, LAPACK's solve): the pose to 1e-9 and the same
    failure reason."""
    import oracle.frontend_np as o
    from oracle import c_oracle as co
    from test_stereo_posit import REASONS, make_problems
    cams = _cams(cam_name)
    P_l, P_r = np.asarray(cams[0].P).reshape(3, 4), np.asarray(cams[1].P).reshape(3, 4)
    seen = set()
    for p in make_problems(cams, seed):
        res = co.solve_stereo_posit(P_l, P_r, p["xyz"], p["uvl"], p["uvr"], p["T_est"], p["T_last"], p["t_imu"])
        T_ref, why = o.solve_stereo_posit(P_l, P_r, p["T_last"], p["t_imu"], p["T_est"], list(zip(p["xyz"], p["uvl"], p["uvr"])))
        seen.add(why)
        assert REASONS.index(why) == res["outcome"], (p["name"], why, res)
        if why is None:
            np.testing.assert_allclose(res["T"][:3], T_ref[:3], rtol=0, atol=1e-9, err_msg=p["name"])
    assert seen == set(REASONS), seen


# ---------------------------------------------------------------------------------------------------------- the sequences
def _static_frames(cams, n, seed=5):
    """A camera that does not move: the same world rendered n times with fresh sensor noise (the regional route and the
    translation clamp)."""
    from svi_mapper_b200.sequence import _render, make_world
    W, H = cams[0].width, cams[0].height
    P_l, P_r = np.asarray(cams[0].P, np.float64).reshape(3, 4), np.asarray(cams[1].P, np.float64).reshape(3, 4)
    planes = make_world(cams[0], 4000)
    rng = np.random.default_rng(seed)
    L = np.stack([_render(planes, P_l, 0.0, np.eye(4), W, H, rng) for _ in range(n)])
    R = np.stack([_render(planes, P_r, -P_r[0, 3] / P_r[0, 0], np.eye(4), W, H, rng) for _ in range(n)])
    return L, R


def _c3_frames(cams, idx, seed=4000):
    """Frames idx of the C3 trajectory (render_sequence's world and camera path), each with its own sensor noise, so that any
    selection of frames can be rendered alone."""
    from svi_mapper_b200.sequence import _render, make_world, smooth_trajectory
    W, H = cams[0].width, cams[0].height
    P_l, P_r = np.asarray(cams[0].P, np.float64).reshape(3, 4), np.asarray(cams[1].P, np.float64).reshape(3, 4)
    planes = make_world(cams[0], seed)
    T = smooth_trajectory(max(idx) + 1, seed)
    frames = {t: (_render(planes, P_l, 0.0, T[t], W, H, np.random.default_rng(2 * t)),
                  _render(planes, P_r, -P_r[0, 3] / P_r[0, 0], T[t], W, H, np.random.default_rng(2 * t + 1))) for t in sorted(set(idx))}
    return np.stack([frames[t][0] for t in idx]), np.stack([frames[t][1] for t in idx]), T[idx]


def _scenarios(cams):
    """name -> (L, R, ground-truth WORLD->LEFT poses or None) of the sequences the tracker runs on."""
    dropped = list(range(8)) + list(range(16, 40, 2))   # eight frames skipped, then every other one: the velocity prior is wrong twice
    far = list(range(8)) + [110, 8, 9, 10]               # one frame 2.5 m ahead: a few stage-2 hits, both solves fail, then back
    L, R, T = _c3_frames(cams, list(range(24)) + dropped + far)
    out = {"c3": (L[:24], R[:24], T[:24])}
    Lb, Rb = L[:24].copy(), R[:24].copy()
    Lb[12:15] = 0
    Rb[12:15] = 0
    out["c3 black"] = (Lb, Rb, None)
    out["static"] = _static_frames(cams, 14) + (None,)
    a, b = 24 + len(dropped), 24 + len(dropped) + len(far)
    out["c3 dropped"] = (L[24:a], R[24:a], T[24:a])
    out["c3 one frame far ahead"] = (L[a:b], R[a:b], None)
    return out


def _pose_error(T, T_gt):
    c_est, c_gt = -T[:3, :3].T @ T[:3, 3], -T_gt[:3, :3].T @ T_gt[:3, 3]
    Rr = T[:3, :3] @ T_gt[:3, :3].T
    return float(np.linalg.norm(c_est - c_gt)), float(np.degrees(np.arccos(np.clip((np.trace(Rr) - 1.0) / 2.0, -1.0, 1.0))))


def test_restated_tracker_tracks_the_c3_sequence():
    """TrackerSV alone, over the C restatement of the front-end: on 24 rendered C3 frames with no pose given, every frame after
    the first takes its pose from the stereo solve and the last pose is within 10 cm and 1 degree of the ground truth -- the
    restatement is a working tracker on its own."""
    from oracle import tracker_np as tn
    from svi_mapper_b200.sequence import render_sequence
    cams = _cams()
    L, R, T = render_sequence(cams[0], cams[1], 24, 4000)
    trk = tn.TrackerSV(cams[0], cams[1], _cfg(cams), threads=_threads())
    sources = []
    for t in range(len(L)):
        trk.process(L[t], R[t])
        sources.append(trk.source)
    assert sources[0] == "prior" and all(s == "posit" for s in sources[1:]), sources
    pos, rot = _pose_error(trk.T_w2l_last, T[-1])
    assert pos <= 0.10 and rot <= 1.0, (pos, rot)
    assert trk.detections >= 2 and len(trk.active()) > 300, (trk.detections, len(trk.active()))


@pytest.fixture(scope="module")
def scenarios():
    return _scenarios(_cams())


# ------------------------------------------------------------------------------------------------------------ GPU: the frame
def _assert_frame_equal(got, want, name):
    """Every output of svi_track_frame_stereo_only byte for byte: source, pose, every field of every solve attempt, the problem
    sizes, the route and both per-landmark results (status and stage first, then the hit fields, then the rest)."""
    assert got["source"] == want["source"], (name, got["source"], want["source"])
    assert got["measurements"] == want["measurements"], (name, got["measurements"], want["measurements"])
    assert len(got["attempts"]) == len(want["attempts"]), name
    for a, b in zip(got["attempts"], want["attempts"]):
        assert [a[k] for k in POSIT_KEYS] == [b[k] for k in POSIT_KEYS], (name, a, b)
        assert a["T"].tobytes() == b["T"].tobytes(), (name, a["T"], b["T"])
    assert got["T"].tobytes() == want["T"].tobytes(), name
    assert got["route"].tobytes() == want["route"].tobytes(), (name, np.flatnonzero(got["route"] != want["route"])[:10])
    for part in ("pose_stage", "epipolar_stage"):
        g, w = got[part], want[part]
        for k in ("status", "stage"):
            assert g[k].tobytes() == w[k].tobytes(), (name, part, k, np.flatnonzero(g[k] != w[k])[:10])
        hit = w["stage"] > 0
        for k in TRACK_KEYS[2:]:
            assert g[k][hit].tobytes() == w[k][hit].tobytes(), (name, part, k, "hits")
        for k in TRACK_KEYS[2:]:
            assert g[k].tobytes() == w[k].tobytes(), (name, part, k, "misses")


def _frame_cases(fe, cams):
    """The cases of test_sv_frame (good prior, mixed flags, prior 3 m off, black frames, regional from the start, n = 0, 25 / 26
    pose hits), then a state of more than 2100 landmarks (C3 states side by side: landmarks are independent) -- three and more
    passes of the 1024-key compaction, a pose problem of many 256-measurement chunks -- with flag patterns whose last candidate
    sits at index 1023, 1024 and 1025, all candidates, none, all leaving, and n = 1."""
    from test_sv_frame import _c3_state, _cases
    L, R, T, st = _c3_state(fe, cams, 9)
    rng = np.random.default_rng(7)
    yield from _cases(fe, L, R, T, st, rng)
    k, s = len(T) - 1, 1.2
    n = len(st["uid"])
    reps = -(-2100 // n) + 1
    big = {kk: np.concatenate([v] * reps) for kk, v in st.items()}
    N = len(big["uid"])
    assert N > 2100
    args = (T[k], T[k - 1], T[k - 1], np.zeros(3), s)
    yield f"n = {N}, all candidates", L[k], R[k], big, np.ones(N, np.uint8), *args
    yield f"n = {N}, mixed flags", L[k], R[k], big, rng.choice(np.array([0, 1, 2, 3], np.uint8), N, p=[0.15, 0.7, 0.1, 0.05]), *args
    yield f"n = {N}, prior 3 m off", L[k], R[k], big, np.ones(N, np.uint8), T[k] + np.pad(np.array([[3.0], [0], [0]]), ((0, 1), (3, 0))), T[k], T[k - 1], np.zeros(3), s
    for last in (1023, 1024, 1025):
        f = np.zeros(N, np.uint8)
        f[: last + 1: 2] = 1          # every other landmark up to the last candidate
        f[last] = 1
        f[last + 1:: 7] = 2           # some of the rest leave
        yield f"last candidate at {last}", L[k], R[k], big, f, *args
    yield f"n = {N}, no candidate", L[k], R[k], big, np.zeros(N, np.uint8), *args
    yield f"n = {N}, all leaving", L[k], R[k], big, np.full(N, 2, np.uint8), *args
    one = {kk: v[:1] for kk, v in st.items()}
    yield "n = 1", L[k], R[k], one, np.ones(1, np.uint8), *args


@pytest.mark.gpu
def test_fused_frame_equals_restated_frame():
    """svi_track_frame_stereo_only against oracle/tracker_np.sv_frame -- the C tracking cascade on the candidate, epipolar and
    regional subsets and the C port of the solve, the routing written out landmark by landmark -- byte for byte on every output,
    on the cases of _frame_cases.  Each source and the routes pose, epipolar, regional and dropped occur."""
    from oracle import tracker_np as tn
    from test_sv_frame import fused
    cams = _cams()
    cfg = _cfg(cams)
    sources, routes, sizes = set(), set(), []
    with StereoFrontend(*cams, max_corners=4000) as fe:
        for name, L, R, st, flags, *rest in _frame_cases(fe, cams):
            got = fused(fe, L, R, st, flags, *rest)
            want = tn.sv_frame(cfg, L, R, st, flags, *rest, threads=_threads())
            _assert_frame_equal(got, want, name)
            sources.add(got["source"])
            routes.update(np.unique(got["route"]).tolist())
            sizes.append(max(got["measurements"]))
            if name == "prior 3 m off":
                assert got["source"] == "posit-damped", got["attempts"]
            if name.startswith("last candidate"):
                assert int(name.split()[-1]) == np.flatnonzero(flags & 1)[-1]
    assert sources == {"posit", "posit-damped", "prior"}, sources
    assert {tn.ROUTE_POSE, tn.ROUTE_EPIPOLAR, tn.ROUTE_REGIONAL, tn.ROUTE_DROPPED} <= routes, routes
    assert max(sizes) > 3 * 256, sizes


# --------------------------------------------------------------------------------------------------------- GPU: the sequences
def _run_demo(tmp_path, name, L, R, mc=4000):
    tag = name.replace(" ", "_")
    Lp, Rp, out = tmp_path / f"{tag}_L.raw", tmp_path / f"{tag}_R.raw", tmp_path / f"{tag}.txt"
    np.ascontiguousarray(L).tofile(Lp)
    np.ascontiguousarray(R).tofile(Rp)
    env = dict(os.environ)
    env.pop("SVI_HOST_POSIT", None)
    env.pop("SVI_HOST_OPTIMIZE", None)
    r = subprocess.run([str(EXE), "--sequence-sv", str(CALIB / "vi_sensor_left.txt"), str(CALIB / "vi_sensor_right.txt"), str(len(L)), str(Lp), str(Rp),
                        str(mc), str(out)], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    frames = []
    for line in out.read_text().splitlines():
        w = line.split()
        if w[0] == "F":
            frames.append(dict(head=w[2:-13], T=w[-12:], M=[], A=[]))
        else:
            frames[-1][w[0]].append(w[1:])
    return frames


def _g(v):
    return "%.17g" % float(v)


def _f(v):
    return "%.9g" % float(v)


def _expected_frame(trk):
    head = ["POSE", trk.source, "VISIBLE", str(trk.visible_last), "ACTIVE", str(len(trk.active())), "S1", str(trk.tracks[0]), "S2", str(trk.tracks[1]),
            "S3", str(trk.tracks[2]), "S22", str(trk.tracks[3]), "DETECTIONS", str(trk.detections), "INSTABILITY", str(trk.instability),
            "POSIT", str(trk.posit_last)]
    T = [_g(trk.T_w2l_last[r, c]) for r in range(3) for c in range(4)]
    M = []
    for lm in trk.visible:
        m = lm.measurements[-1]
        M.append([str(lm.uid), _f(m[2][0]), _f(m[2][1]), _f(m[3][0]), _f(m[3][1])] + [_g(v) for v in lm.last_xyz_left])
    A = [[str(lm.uid)] + [_g(v) for v in lm.xyz_opt] + [str(int(lm.optimal)), str(int(lm.visible)), str(lm.opt_success), str(lm.opt_failed),
                                                       str(lm.failed), str(len(lm.measurements))] for lm in trk.active()]
    return dict(head=head, T=T, M=M, A=A)


def _lockstep(tmp_path, name, L, R):
    """facade_demo --sequence-sv (the fused frame call) and TrackerSV over the same frames, compared frame by frame; returns what
    occurred along the way."""
    from oracle import tracker_np as tn
    cams = _cams()
    frames = _run_demo(tmp_path, name, L, R)
    assert len(frames) == len(L)
    trk = tn.TrackerSV(cams[0], cams[1], _cfg(cams), threads=_threads())
    seen = dict(sources=set(), routes=set(), retired=0, optimisation_failures=0, failed_solves_with_hits=0)
    for t in range(len(L)):
        before = {lm.uid for lm in trk.active()}
        trk.process(L[t], R[t])
        got, want = frames[t], _expected_frame(trk)
        assert got["head"] == want["head"], (name, t, got["head"], want["head"])
        assert got["T"] == want["T"], (name, t, got["T"], want["T"])
        assert [m[0] for m in got["M"]] == [m[0] for m in want["M"]], (name, t)
        for a, b in zip(got["M"], want["M"]):
            assert a == b, (name, t, a, b)
        assert [a[0] for a in got["A"]] == [a[0] for a in want["A"]], (name, t)
        for a, b in zip(got["A"], want["A"]):
            assert a == b, (name, t, a, b)
        seen["sources"].add(trk.source)
        seen["routes"].update(np.unique(trk.last["route"]).tolist())
        seen["retired"] += len(before - {lm.uid for lm in trk.active()})
        seen["optimisation_failures"] += sum(1 for lm in trk.active() if lm.opt_failed > 0) if t % 10 == 0 else 0
        seen["failed_solves_with_hits"] += sum(1 for a, m in zip(trk.last["attempts"], trk.last["measurements"]) if a["outcome"] != 0 and m > 0)
    return seen, trk


@pytest.mark.gpu
def test_cpp_tracker_sequences_match_restated_tracker(tmp_path, scenarios):
    """facade_demo --sequence-sv (CTrackerSV over svi_track_frame_stereo_only and svi_optimize_landmarks) in lockstep with
    oracle/tracker_np.TrackerSV over the C restatement, frame by frame: the F line (pose source, visible, active, the four stage
    counters, detections, instability, problem size of the last accepted solve and the 12 numbers of the pose), every M line
    (landmark, both image points, the triangulated point) and every A line (landmark, optimised position, optimal, visible,
    optimisation successes and failures, failed trackings, measurements), all as printed -- exact, the optimised positions too:
    both sides refine landmarks with solvers that equal the host's loop bit for bit.  Scenarios: 24 C3 frames; the same with
    three black frames (prior source, instability, recovery); a static camera (regional route, translation clamp); C3 with
    skipped frames (a wrong constant-velocity prior); C3 with one frame from 2.5 m further on (solves that fail on a handful of
    hits, whose landmarks must get no measurement).  Across them: the sources posit and prior, the routes pose, epipolar, regional
    and dropped, a retired landmark, an optimisation round that leaves landmarks with failed optimisations, and failed solves
    that had measurements.  No rendered scenario reaches posit-damped: the stage-2 search around a wrong constant-velocity prior
    still finds far more than 25 points on the distant cards, and the solve converges from there; the damped retry is covered
    by test_fused_frame_equals_restated_frame ("prior 3 m off").  The no-translation re-route cannot occur behind the device's
    split (see sv_scatter_kernel)."""
    total = dict(sources=set(), routes=set(), retired=0, optimisation_failures=0, failed_solves_with_hits=0)
    for name, (L, R, T_gt) in scenarios.items():
        seen, trk = _lockstep(tmp_path, name, L, R)
        for k in ("sources", "routes"):
            total[k] |= seen[k]
        for k in ("retired", "optimisation_failures", "failed_solves_with_hits"):
            total[k] += seen[k]
        if name == "c3":
            assert _pose_error(trk.T_w2l_last, T_gt[-1])[0] <= 0.10
    assert {"posit", "prior"} <= total["sources"], total
    assert {1, 2, 3, 5} <= total["routes"], total
    assert total["retired"] > 0 and total["optimisation_failures"] > 0 and total["failed_solves_with_hits"] > 0, total


@pytest.mark.gpu
def test_bounds_checked_build_tracker_sv_oracle(tmp_path):
    """The GPU tests of this file once against the -DSVI_BOUNDS_CHECK build (every run-time index of the frame call's kernels
    asserted; a failed assertion fails the call): the Python binding loads it through SVI_GPU_LIB, facade_demo finds it as
    libsvi_gpu.so on LD_LIBRARY_PATH, which comes before its RUNPATH."""
    import shutil
    from svi_mapper_b200 import build as bld
    lib = bld.build_checked()
    libdir = tmp_path / "checked"
    libdir.mkdir()
    shutil.copy(lib, libdir / "libsvi_gpu.so")
    env = dict(os.environ, SVI_GPU_LIB=str(lib), LD_LIBRARY_PATH=os.pathsep.join(filter(None, [str(libdir), os.environ.get("LD_LIBRARY_PATH")])))
    r = subprocess.run([sys.executable, "-m", "pytest", str(pathlib.Path(__file__)), "-x", "-q", "-m", "gpu", "-k", "restated"], env=env,
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "2 passed" in r.stdout and "failed" not in r.stdout
