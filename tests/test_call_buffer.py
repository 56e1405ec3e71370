"""The call buffer of libsvi_gpu (DESIGN.md section 3): the per-query, tracking and solver entry points stage their arrays
through one device block and its pinned mirror, which grows when a call needs more.  Every user runs on one shared context in
shuffled orders while the buffer grows under them, on a context whose max_queries is past the buffer's initial cap, and at
the capacity bound of the two matchers; each result must equal, byte for byte, the same call on a fresh default context."""
import pathlib

import numpy as np
import pytest

from svi_mapper_b200 import StereoFrontend, load_camera
from svi_mapper_b200.frontend import SviError

CALIB = pathlib.Path(__file__).resolve().parent / "golden" / "calib"

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("built_library")]


@pytest.fixture(scope="module")
def cams():
    return load_camera(str(CALIB / "vi_sensor_left.txt")), load_camera(str(CALIB / "vi_sensor_right.txt"))


@pytest.fixture(scope="module")
def c3(cams):
    """The last frame of a short C3 sequence and the SequenceTracker's landmark state before it (true poses)."""
    from svi_mapper_b200.sequence import GpuBackend, SequenceTracker, render_sequence
    L, R, T = render_sequence(cams[0], cams[1], 9, 4000)
    with StereoFrontend(*cams, max_corners=4000) as fe:
        trk = SequenceTracker(GpuBackend(fe), cams[0])
        for t in range(len(T) - 1):
            trk.process(L[t], R[t], T[t])
        st = {k: v.copy() for k, v in trk.s.items()}
    assert len(st["uid"]) > 300
    return L[-1], R[-1], T[-1], T[-2], st


def _flat(r):
    """Every array of a result, in a fixed order, as bytes."""
    if isinstance(r, dict):
        return [b for k in sorted(r) for b in _flat(r[k])]
    if isinstance(r, (list, tuple)):
        return [b for v in r for b in _flat(v)]
    if isinstance(r, np.ndarray):
        return [r.tobytes()]
    return [repr(r).encode()]


def _optimize_args(cams, n, per, rng):
    """n landmarks with `per` stereo measurements each over 8 poses."""
    P_l, P_r = (np.asarray(c.P, np.float64).reshape(3, 4) for c in cams)
    T = np.stack([np.eye(4)] * 8)
    T[:, :3, 3] = np.stack([0.1 * np.arange(8), np.zeros(8), 0.05 * np.arange(8)], 1)
    proj_l, proj_r = P_l @ T, P_r @ T
    xyz = rng.uniform([-3.0, -2.0, 4.0], [3.0, 2.0, 12.0], (n, 3))
    pose = rng.integers(0, 8, n * per).astype(np.int32)
    pts = np.c_[np.repeat(xyz, per, 0), np.ones(n * per)]
    uv = lambda P: (lambda h: (h[:, :2] / h[:, 2:]).astype(np.float32))(np.einsum("kij,kj->ki", P[pose], pts))
    noise = lambda: rng.normal(0.0, 0.3, (n * per, 2)).astype(np.float32)
    guess = xyz + rng.normal(0.0, 0.05, (n, 3))
    return guess, np.arange(n + 1, dtype=np.int32) * per, pose, uv(proj_l) + noise(), uv(proj_r) + noise(), proj_l, proj_r


def _posit_args(cams, n, rng):
    P_l, P_r = (np.asarray(c.P, np.float64).reshape(3, 4) for c in cams)
    T = np.eye(4)
    T[:3, 3] = [0.2, -0.1, 0.3]
    xyz = rng.uniform([-4.0, -2.0, 3.0], [4.0, 2.0, 15.0], (n, 3))
    h = lambda P: P @ T @ np.c_[xyz, np.ones(n)].T
    uv = lambda P: (lambda q: (q[:2] / q[2]).T.astype(np.float32))(h(P))
    prior = T.copy()
    prior[:3, 3] += [0.02, 0.0, -0.02]
    return xyz, uv(P_l) + rng.normal(0, 0.5, (n, 2)).astype(np.float32), uv(P_r) + rng.normal(0, 0.5, (n, 2)).astype(np.float32), prior


def _calls(cams, c3, n):
    """(name, call(fe)) for every user of the call buffer; per-landmark calls on the first n landmarks of the C3 state."""
    L, R, T, T_prev, st = c3
    W, H = cams[0].width, cams[0].height
    rng = np.random.default_rng(11)
    s = {k: v[:n] for k, v in st.items()}
    xy = np.stack([rng.integers(28, W - 28, n), rng.integers(28, H - 28, n)], 1).astype(np.float32)
    with StereoFrontend(*cams) as fe:
        desc_l, _ = fe.describe(L, xy)
        desc_r, _ = fe.describe(R, xy)
    rng_f = rng.uniform(0.5, 90.0, n).astype(np.float32)
    tl_r = np.stack([np.maximum(0, xy[:, 0] - 28 - rng_f), xy[:, 1] - 28], 1).astype(np.float32)
    tl_l = np.stack([xy[:, 0] - 28, xy[:, 1] - 28], 1).astype(np.float32)
    q = rng.integers(0, 256, (3000, 32), dtype=np.uint8)
    t = rng.integers(0, 256, (2500, 32), dtype=np.uint8)
    qxy = rng.uniform(0, [W, H], (3000, 2)).astype(np.float32)
    txy = rng.uniform(0, [W, H], (2500, 2)).astype(np.float32)
    opt = _optimize_args(cams, 20000, 6, rng)    # ~3.7 MB: more than the buffer of max_queries = 64 holds at creation
    posit = _posit_args(cams, 3000, rng)
    ref = dict(uv_reference_left=s["uv_ref"], desc_reference_left=s["ref_desc_l"], T_left_to_world_at_detection=s["T_det"])
    track = lambda fe, **kw: fe.track_landmarks(L, R, T, s["xyz_w"], s["last_desc_l"], s["last_desc_r"], s["last_disp"], 7.0, 1.2, **kw)
    return [
        ("describe", lambda fe: fe.describe(L, xy)),
        ("triangulate_right", lambda fe: fe.triangulate_right(R, tl_r, xy, desc_l)),
        ("triangulate_left", lambda fe: fe.triangulate_left(L, rng_f, tl_l, xy, desc_r)),
        ("point_in_left", lambda fe: fe.point_in_left(xy, xy - np.float32([12.5, 0.0]))),
        ("match_hamming", lambda fe: fe.match_hamming(q, t)),
        ("match_hamming no train", lambda fe: fe.match_hamming(q[:50], t[:0])),
        ("match_epipolar", lambda fe: fe.match_epipolar(q, qxy, t, txy, 2.0, 0.0, 200.0)),
        ("mask", lambda fe: fe.mask_active_landmarks(xy)),
        ("stereo_frame_masked", lambda fe: fe.add_new_landmarks(L, R, mask_centres=xy)),
        ("track_landmarks", lambda fe: track(fe, **ref)),
        ("track_landmarks stages 1-2", lambda fe: track(fe, stages=3)),
        ("optimize_landmarks", lambda fe: fe.optimize_landmarks(*opt)),
        ("solve_stereo_posit", lambda fe: fe.solve_stereo_posit(*posit)),
        ("track_frame_stereo_only", lambda fe: fe.track_frame_stereo_only(L, R, s["xyz_w"], s["last_desc_l"], s["last_desc_r"], s["last_disp"], 7.0,
                                                                         s["uv_ref"], s["ref_desc_l"], s["T_det"], np.ones(n, np.uint8), T, T_prev,
                                                                         T_prev, np.zeros(3), 1.2)),
    ]


def _fresh(cams, call):
    with StereoFrontend(*cams) as fe:
        return _flat(call(fe))


def test_every_user_shares_one_growing_buffer(cams, c3):
    """On one context with max_queries = 64 every user runs in two seeded shuffled orders; optimize_landmarks needs more than
    the buffer holds, so it grows part-way through the first pass.  Each result equals the call on a fresh default context."""
    calls = _calls(cams, c3, 64)
    want = {name: _fresh(cams, call) for name, call in calls}
    rng = np.random.default_rng(5)
    with StereoFrontend(*cams, max_queries=64) as fe:
        for rep in range(2):
            for i in rng.permutation(len(calls)):
                name, call = calls[i]
                assert _flat(call(fe)) == want[name], (rep, name)


def test_large_max_queries(cams, c3):
    """max_queries = 150000 puts the buffer's creation size past its 64 MiB cap: describe, the hamming matcher and the full
    tracking call still give what a default context gives."""
    calls = dict(_calls(cams, c3, len(c3[4]["uid"])))
    with StereoFrontend(*cams, max_queries=150000) as fe:
        for name in ("describe", "match_hamming", "track_landmarks"):
            assert _flat(calls[name](fe)) == _fresh(cams, calls[name]), name


def test_match_capacity_bound(cams):
    """The matchers refuse inputs past max_queries * 512 + max_corners * 64 + 3 * W * H + 1 MiB bytes at 40 (hamming) and
    48 + 16 per query (epipolar) bytes per descriptor, one element past the bound and not at it."""
    W, H = cams[0].width, cams[0].height
    with StereoFrontend(*cams, max_queries=64) as fe:
        bound = 64 * 512 + fe.max_corners * 64 + 3 * W * H + (1 << 20)
        q = np.zeros((1, 32), np.uint8)
        n_ok = bound // 40 - 1
        fe.match_hamming(q, np.zeros((n_ok, 32), np.uint8))
        with pytest.raises(SviError, match="svi_match_hamming: raise max_queries"):
            fe.match_hamming(q, np.zeros((n_ok + 1, 32), np.uint8))
        n_ok = (bound - 16) // 48 - 1
        qxy = np.zeros((1, 2), np.float32)
        fe.match_epipolar(q, qxy, np.zeros((n_ok, 32), np.uint8), np.zeros((n_ok, 2), np.float32))
        with pytest.raises(SviError, match="svi_match_epipolar: raise max_queries"):
            fe.match_epipolar(q, qxy, np.zeros((n_ok + 1, 32), np.uint8), np.zeros((n_ok + 1, 2), np.float32))
