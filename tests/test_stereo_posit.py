"""The pose solve of the stereo-only tracker (CSolverStereoPosit::getTransformationWORLDtoLEFT, reference
src/optimization/CSolverStereoPosit.cpp:8-170) on the GPU: svi_solve_stereo_posit against the C++ host layer's CPU loop bit for
bit, the CPU loop against the numpy restatement, and CTrackerSV (facade_demo --sequence-sv) recovering the trajectory of a
rendered moving sequence without any ground-truth pose."""
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

pytestmark = pytest.mark.usefixtures("built_library")

SIZES = (26, 31, 32, 33, 255, 256, 257, 1000, 4000)
REASONS = (None, "insufficient number of points", "insufficient accuracy", "inconsistent with prior")


def _rot(ax, ang):
    ax = np.asarray(ax, float) / np.linalg.norm(ax)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    return np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K


def _pose(ax, ang, t):
    T = np.eye(4)
    T[:3, :3] = _rot(ax, ang)
    T[:3, 3] = t
    return T


def _observe(P_l, P_r, T, xyz, rng, noise=0.3):
    """stereo image points of WORLD points xyz seen from WORLD->LEFT pose T, float32 with pixel noise"""
    q = np.c_[xyz @ T[:3, :3].T + T[:3, 3], np.ones(len(xyz))]
    a, b = q @ P_l.T, q @ P_r.T
    uvl = (a[:, :2] / a[:, 2:]).astype(np.float32) + rng.normal(0, noise, (len(xyz), 2)).astype(np.float32)
    uvr = np.c_[b[:, 0] / b[:, 2], uvl[:, 1]].astype(np.float32)
    uvr[:, 0] += rng.normal(0, noise, len(xyz)).astype(np.float32)
    return uvl, uvr


def make_problems(cams, seed):
    """Seeded problems for one stereo camera: every size of SIZES with a perturbed prior, outliers and points behind the
    camera, the translation clamp, and one problem per failure that a finite input reaches.  Each: dict(name, xyz, uvl, uvr, T_est, T_last, t_imu)."""
    P_l, P_r = np.asarray(cams[0].P, np.float64).reshape(3, 4), np.asarray(cams[1].P, np.float64).reshape(3, 4)
    rng = np.random.default_rng(seed)
    probs = []

    def scene(n):
        return np.c_[rng.uniform(-4, 4, n), rng.uniform(-2, 2, n), rng.uniform(3, 25, n)]

    for k, n in enumerate(SIZES):
        T_true = _pose(rng.normal(size=3), rng.uniform(0.0, 0.05), rng.normal(0, 0.1, 3))
        xyz = scene(n)
        uvl, uvr = _observe(P_l, P_r, T_true, xyz, rng)
        out = rng.random(n) < 0.1                                # outliers: down-weighted, not rejected
        uvl[out] += rng.uniform(-40, 40, (int(out.sum()), 2)).astype(np.float32)
        behind = rng.random(n) < 0.05                           # points behind the camera: no contribution, still counted
        xyz[behind, 2] = -rng.uniform(1, 5, int(behind.sum()))
        T_est = _pose(rng.normal(size=3), 0.02, [0.0, 0.0, 0.0]) @ T_true
        T_est[:3, 3] += rng.normal(0, 0.05, 3)
        T_last = _pose([0, 1, 0], 0.01 * k, rng.normal(0, 0.2, 3))
        probs.append(dict(name=f"n{n}", xyz=xyz, uvl=uvl, uvr=uvr, T_est=T_est, T_last=T_last, t_imu=rng.normal(0, 0.05, 3)))
    # translation clamp: the solution lands within sqrt(0.001) m of T_last, whose translation it keeps
    T_true = _pose([0.3, 1, 0], 0.02, [0.05, -0.02, 0.3])
    xyz = scene(300)
    uvl, uvr = _observe(P_l, P_r, T_true, xyz, rng)
    T_last = T_true.copy()
    T_last[:3, 3] += [0.012, -0.008, 0.015]
    probs.append(dict(name="clamp", xyz=xyz, uvl=uvl, uvr=uvr, T_est=np.eye(4), T_last=T_last, t_imu=np.zeros(3)))
    # too few points
    probs.append(dict(name="n25", xyz=xyz[:25], uvl=uvl[:25], uvr=uvr[:25], T_est=np.eye(4), T_last=np.eye(4), t_imu=np.zeros(3)))
    probs.append(dict(name="n0", xyz=xyz[:0], uvl=uvl[:0], uvr=uvr[:0], T_est=T_true, T_last=np.eye(4), t_imu=np.zeros(3)))
    # insufficient accuracy: nearly every measurement far off
    T_true = _pose([1, 0.2, 0], 0.01, [0.02, 0.01, 0.05])
    xyz = scene(40)
    uvl, uvr = _observe(P_l, P_r, T_true, xyz, rng)
    uvl[2:] += rng.choice([-1, 1], (38, 2)).astype(np.float32) * rng.uniform(60, 150, (38, 2)).astype(np.float32)
    probs.append(dict(name="inaccurate", xyz=xyz, uvl=uvl, uvr=uvr, T_est=np.eye(4), T_last=np.eye(4), t_imu=np.zeros(3)))
    # high risk: the measurements put the camera 2.5 m from the prior
    xyz = scene(80)
    uvl, uvr = _observe(P_l, P_r, _pose([0, 1, 0], 0.0, [2.5, 0, 0]), xyz, rng, noise=0.0)
    probs.append(dict(name="risk", xyz=xyz, uvl=uvl, uvr=uvr, T_est=np.eye(4), T_last=np.eye(4), t_imu=np.zeros(3)))
    # (no problem here reaches the 1000-iteration cap: a singular system turns the pose into NaN, every point then drops out
    # behind the camera, the total error is 0 twice in a row and the loop "converges" -- on a NaN pose, whose sign bit differs
    # between the x86 default NaN and the GPU's, so such a problem has no bit-exact printed form to compare)
    return probs


def _write_problem(path, p):
    rows = [" ".join(repr(float(v)) for v in np.concatenate([np.ravel(p["T_est"]), np.ravel(p["T_last"]), np.ravel(p["t_imu"])]))]
    rows += [" ".join([repr(float(v)) for v in x] + [repr(float(v)) for v in a] + [repr(float(v)) for v in b]) for x, a, b in zip(p["xyz"], p["uvl"], p["uvr"])]
    path.write_text("\n".join(rows) + "\n")


def _demo_posit(cam_name, p, tmp_path, mode):
    f = tmp_path / f"{p['name']}.txt"
    _write_problem(f, p)
    env = dict(os.environ)
    env.pop("SVI_HOST_POSIT", None)
    if mode == "cpu":
        env["SVI_HOST_POSIT"] = "cpu"
    r = subprocess.run([str(EXE), "--posit", str(CALIB / f"{cam_name}_left.txt"), str(CALIB / f"{cam_name}_right.txt"), str(f)],
                       capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    return r.stdout.strip()


def _cams(name):
    from svi_mapper_b200 import load_camera
    return load_camera(str(CALIB / f"{name}_left.txt")), load_camera(str(CALIB / f"{name}_right.txt"))


def _expected_line(res, n):
    """What facade_demo --posit prints for a result of the binding (the C++ host's what() texts, std::to_string = %f)."""
    oc = res["outcome"]
    if oc == _lib.SVI_POSIT_OK:
        return " ".join("%.17g" % v for v in res["T"][:3].ravel()) + " %d" % res["iterations"]
    if oc == _lib.SVI_POSIT_TOO_FEW_POINTS:
        return "FAILED insufficient number of points: %d" % n
    if oc == _lib.SVI_POSIT_INACCURATE:
        return "FAILED insufficient accuracy (average error: %f inliers: %d)" % (res["average_squared_error"], res["inliers"])
    if oc == _lib.SVI_POSIT_HIGH_RISK:
        return "FAILED inconsistent with prior (HIGH RISK: %f)" % res["risk"]
    return "FAILED system did not converge"


def test_solve_stereo_posit_rejects_a_null_context():
    import ctypes as C
    lib = _lib.load()
    assert lib.svi_solve_stereo_posit(None, C.byref(_lib.PositProblem()), C.byref(_lib.PositResult())) == _lib.SVI_ERR_INVALID
    assert lib.svi_solve_stereo_posit(None, None, None) == _lib.SVI_ERR_INVALID


@pytest.mark.parametrize("cam_name,seed", [("vi_sensor", 21), ("kitti_11_12", 22)])
def test_host_cpu_loop_matches_oracle_with_priors(cam_name, seed, tmp_path):
    """facade_demo --posit under SVI_HOST_POSIT=cpu (the C++ host's CPU loop, no GPU) against oracle.frontend_np.solve_stereo_posit
    on the seeded problem set -- non-identity priors, outliers, points behind the camera, the clamp and the failures: the
    pose to 1e-9 and the same failure reason."""
    import oracle.frontend_np as o
    cams = _cams(cam_name)
    P_l, P_r = np.asarray(cams[0].P).reshape(3, 4), np.asarray(cams[1].P).reshape(3, 4)
    seen = set()
    for p in make_problems(cams, seed):
        line = _demo_posit(cam_name, p, tmp_path, "cpu")
        T_ref, why = o.solve_stereo_posit(P_l, P_r, p["T_last"], p["t_imu"], p["T_est"], list(zip(p["xyz"], p["uvl"], p["uvr"])))
        seen.add(why)
        if why is None:
            v = line.split()
            assert len(v) == 13, (p["name"], line)
            np.testing.assert_allclose(np.array([float(t) for t in v[:12]]).reshape(3, 4), T_ref[:3], rtol=0, atol=1e-9, err_msg=p["name"])
            if p["name"] == "clamp":
                assert [float(t) for t in v[3:12:4]] == list(p["T_last"][:3, 3]), line
        else:
            assert line.startswith("FAILED " + why), (p["name"], line, why)
    assert seen == set(REASONS), seen


@pytest.mark.gpu
def test_gpu_solve_is_bit_identical_to_host_loop(tmp_path):
    """svi_solve_stereo_posit through the Python binding and through the C++ host layer (facade_demo --posit) against the host's
    CPU loop (SVI_HOST_POSIT=cpu): all 12 numbers to the last digit, the iteration count and every FAILED text, on vi_sensor and
    kitti_11_12, in two orders on one ctx (staging buffer growth and shrink), interleaved with svi_optimize_landmarks calls that
    share the staging buffer."""
    for cam_name, seed in (("vi_sensor", 31), ("kitti_11_12", 32)):
        cams = _cams(cam_name)
        probs = make_problems(cams, seed)
        want = {p["name"]: _demo_posit(cam_name, p, tmp_path, "cpu") for p in probs}
        outcomes = set()
        for p in probs:
            assert _demo_posit(cam_name, p, tmp_path, "gpu") == want[p["name"]], (cam_name, p["name"])
        P_l, P_r = np.asarray(cams[0].P).reshape(3, 4), np.asarray(cams[1].P).reshape(3, 4)
        rng = np.random.default_rng(seed)
        with StereoFrontend(*cams) as fe:
            for order in (rng.permutation(len(probs)), rng.permutation(len(probs))[::-1]):
                for k, i in enumerate(order):
                    p = probs[i]
                    res = fe.solve_stereo_posit(p["xyz"], p["uvl"], p["uvr"], p["T_est"], p["T_last"], p["t_imu"])
                    assert _expected_line(res, len(p["xyz"])) == want[p["name"]], (cam_name, p["name"], res)
                    outcomes.add(res["outcome"])
                    if res["outcome"] != _lib.SVI_POSIT_OK:
                        assert np.array_equal(res["T"], np.asarray(p["T_est"], np.float64))
                    if k % 3 == 0:   # a landmark refinement in between: the same staging pair, other sizes
                        m = int(rng.integers(6, 4000))
                        xyz = np.array([[0.2, -0.1, 8.0]])
                        uvl, uvr = _observe(P_l, P_r, np.eye(4), np.repeat(xyz, m, 0), rng)
                        got = fe.optimize_landmarks(xyz + 0.05, [0, m], np.zeros(m, np.int32), uvl, uvr, P_l[None], P_r[None])
                        assert int(got["outcome"][0]) in (_lib.SVI_OPT_CONVERGED, _lib.SVI_OPT_OPTIMAL)
            # the convenience defaults: T_last = T_estimate, t_imu = 0
            p = probs[0]
            a = fe.solve_stereo_posit(p["xyz"], p["uvl"], p["uvr"], p["T_est"])
            b = fe.solve_stereo_posit(p["xyz"], p["uvl"], p["uvr"], p["T_est"], p["T_est"], np.zeros(3))
            assert np.array_equal(a["T"], b["T"]) and a["outcome"] == b["outcome"]
        assert outcomes == {_lib.SVI_POSIT_OK, _lib.SVI_POSIT_TOO_FEW_POINTS, _lib.SVI_POSIT_INACCURATE, _lib.SVI_POSIT_HIGH_RISK}, outcomes


def _sequence_sv(tmp_path, n, mc, mode, seed=4000):
    from svi_mapper_b200.sequence import render_sequence
    cams = _cams("vi_sensor")
    Lp, Rp = tmp_path / "L.raw", tmp_path / "R.raw"
    if not Lp.exists():
        L, R, T = render_sequence(cams[0], cams[1], n, seed)
        L.tofile(Lp)
        R.tofile(Rp)
        np.save(tmp_path / "T.npy", T)
    out = tmp_path / f"sv_{mode}.txt"
    env = dict(os.environ)
    env.pop("SVI_HOST_POSIT", None)
    if mode == "cpu":
        env["SVI_HOST_POSIT"] = "cpu"
    r = subprocess.run([str(EXE), "--sequence-sv", str(CALIB / "vi_sensor_left.txt"), str(CALIB / "vi_sensor_right.txt"), str(n), str(Lp), str(Rp),
                        str(mc), str(out)], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    return out.read_text(), np.load(tmp_path / "T.npy")


def parse_sequence_sv(text):
    frames = []
    for line in text.splitlines():
        w = line.split()
        if w[0] == "F":
            head = dict(zip(w[2:-13:2], w[3:-13:2]))
            T = np.eye(4)
            T[:3] = np.array([float(v) for v in w[-12:]]).reshape(3, 4)
            frames.append(dict(head, T=T))
    return frames


@pytest.mark.gpu
def test_stereo_only_tracker_recovers_the_trajectory(tmp_path):
    """CTrackerSV over 60 rendered frames of the C3 sequence (about 1.5 m of forward motion with sway, yaw and pitch) with no pose
    given: the GPU solve and the host's CPU loop give byte-identical runs, every frame after the first takes its pose from
    the stereo solve, and the recovered WORLD->LEFT pose ends within 10 cm and 1 degree of the ground truth."""
    n, mc = 60, 4000
    gpu, T_gt = _sequence_sv(tmp_path, n, mc, "gpu")
    cpu, _ = _sequence_sv(tmp_path, n, mc, "cpu")
    assert gpu == cpu
    frames = parse_sequence_sv(gpu)
    assert len(frames) == n
    assert frames[0]["POSE"] == "prior"   # no landmarks yet: the first frame keeps the identity prior
    sources = [f["POSE"] for f in frames[1:]]
    assert all(s == "posit" for s in sources), sources
    pos_err, rot_err = [], []
    for f, T in zip(frames, T_gt):
        c_est, c_gt = -f["T"][:3, :3].T @ f["T"][:3, 3], -T[:3, :3].T @ T[:3, 3]
        pos_err.append(float(np.linalg.norm(c_est - c_gt)))
        R = f["T"][:3, :3] @ T[:3, :3].T
        rot_err.append(float(np.degrees(np.arccos(np.clip((np.trace(R) - 1.0) / 2.0, -1.0, 1.0)))))
    path = float(np.linalg.norm(-T_gt[-1][:3, :3].T @ T_gt[-1][:3, 3]))
    print(f"path {path:.3f} m, final position error {pos_err[-1] * 100:.2f} cm (max {max(pos_err) * 100:.2f}), "
          f"final rotation error {rot_err[-1]:.3f} deg (max {max(rot_err):.3f})")
    assert path > 1.4
    assert pos_err[-1] <= 0.10, pos_err
    assert rot_err[-1] <= 1.0, rot_err


@pytest.mark.gpu
def test_bounds_checked_build_stereo_posit():
    """The GPU solve tests of this file once against the -DSVI_BOUNDS_CHECK build: every run-time shared-memory and array index
    of stereo_posit_kernel is asserted there (the Python binding loads that build; facade_demo keeps its own library)."""
    from svi_mapper_b200 import build as bld
    lib = bld.build_checked()
    r = subprocess.run([sys.executable, "-m", "pytest", str(pathlib.Path(__file__)), "-x", "-q", "-m", "gpu", "-k", "bit_identical"],
                       env=dict(os.environ, SVI_GPU_LIB=str(lib)), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "failed" not in r.stdout
