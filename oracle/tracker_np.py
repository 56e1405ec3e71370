"""CPU restatement of the per-frame tracker loops around the stereo front-end -- TEST INFRASTRUCTURE ONLY (tests/ compare
the C++ host layer svi_mapper_b200/host/CTrackerGT.h, CTrackerSV.h + CFundamentalMatcher.h, which drive the GPU, against this).

What it restates (paths relative to the reference tree):
  CTrackerGT::_trackLandmarks                 src/core/CTrackerGT.cpp:137-380  (motion scaling :157, trackManual :167,
                                              optimizeActiveLandmarks :197, re-detection trigger :305-315)
  CFundamentalMatcher::trackManual            src/core/CFundamentalMatcher.cpp:1334-2027 (candidate rule :1375-1395, image work
                                              by oracle/svi_oracle.c, bookkeeping :1980-2009)
  CFundamentalMatcher::addNewLandmarks        :83-193, getMaskActiveLandmarks :2043-2073
  CLandmark::addMeasurement / optimize        src/types/CLandmark.cpp:80-296, :447-581 (frontend_np.optimize_landmark; the
                                              stereo-only tracker uses the bit-exact C port svo_optimize_landmark)
  CTrackerSV::process / _trackLandmarks       src/core/CTrackerSV.cpp:143-172, :234-552 (priors and motion scaling :243-254,
                                              pose fallback :268-313, instability :333-349, optimisation :362-365, re-detection
                                              :468-473, motion update :547-548) -> TrackerSV
  CFundamentalMatcher::getPoseStereoPosit     :338-757 (candidates = optimal landmarks, stages 1-2, CSolverStereoPosit on the hits,
                                              measurements under the solved pose) and trackEpipolar :760-1332 (leave :808-825,
                                              seen :830-833, epipolar / regional split :800, :1804, failures :1014-1023,
                                              :1281-1289, activity :1291-1312) -> sv_frame + TrackerSV
  CSolverStereoPosit::getTransformationWORLDtoLEFT  src/optimization/CSolverStereoPosit.cpp:8-170 (oracle/svi_oracle.c
                                              svo_solve_stereo_posit, the host's CPU loop to the last bit)
Pose algebra is written out element by element in the order the host layer uses, so that both sides see the same doubles."""
from __future__ import annotations

import numpy as np

from . import c_oracle as co
from . import frontend_np as o

ST_EPI_NO_TRANSLATION = 24
MAX_FAILED = 5


def iso_mul(A, B):
    """Isometry3d * Isometry3d of the host layer: rows 0..2, s = ((a0*b0 + a1*b1) + a2*b2) (+ a3 in the last column)."""
    C = np.eye(4)
    for r in range(3):
        for c in range(4):
            s = 0.0
            for k in range(3):
                s += A[r, k] * B[k, c]
            C[r, c] = s + (A[r, 3] if c == 3 else 0.0)
    return C


def iso_inv(T):
    I = np.eye(4)
    for r in range(3):
        for c in range(3):
            I[r, c] = T[c, r]
    for r in range(3):
        I[r, 3] = -(I[r, 0] * T[0, 3] + I[r, 1] * T[1, 3] + I[r, 2] * T[2, 3])
    return I


def iso_apply(T, p):
    return np.array([T[r, 0] * p[0] + T[r, 1] * p[1] + T[r, 2] * p[2] + T[r, 3] for r in range(3)])


def proj_mul(P, T):
    R = np.zeros((3, 4))
    for r in range(3):
        for c in range(4):
            s = 0.0
            for k in range(4):
                s += P[r, k] * T[k, c]
            R[r, c] = s
    return R


class Landmark:
    def __init__(self, uid, desc_l, desc_r, size, uvl, uvr, xyz_left, T_l2w, P_w2l, P_w2r):
        self.uid, self.ref_desc_l, self.size = uid, desc_l.copy(), float(size)
        self.xyz_opt = iso_apply(T_l2w, xyz_left)
        self.uv_ref = np.array([float(uvl[0]), float(uvl[1])])
        self.failed = self.opt_success = self.opt_failed = 0
        self.optimal = self.visible = False
        self.measurements = []
        self.add_measurement(uvl, uvr, desc_l, desc_r, xyz_left, P_w2l, P_w2r)

    def add_measurement(self, uvl, uvr, desc_l, desc_r, xyz_left, P_w2l, P_w2r):
        self.last_desc_l, self.last_desc_r = desc_l.copy(), desc_r.copy()
        self.last_uv_l = (np.float32(uvl[0]), np.float32(uvl[1]))
        self.last_disp = np.float32(np.float32(uvl[0]) - np.float32(uvr[0]))
        self.last_xyz_left = np.asarray(xyz_left, np.float64).copy()
        self.measurements.append((P_w2l, P_w2r, (np.float32(uvl[0]), np.float32(uvl[1])), (np.float32(uvr[0]), np.float32(uvr[1]))))

    def optimize(self):
        self.optimal = False
        r = o.optimize_landmark(self.xyz_opt, self.measurements)
        self.xyz_opt = np.asarray(r["xyz"], np.float64)
        self.optimal = bool(r["optimal"])
        self.opt_success += r["success"]
        self.opt_failed += r["failed"]

    def optimize_exact(self, native=False):
        """CLandmark::optimize :281-296 through svo_optimize_landmark (bit-exact with the host): more than five measurements are
        refined; a converged refinement moves the landmark (optimal when its average error is below 9 px^2), a rejected or
        non-converged one keeps the position and counts as failed; fewer measurements leave it optimal."""
        r = co.optimize_landmark(self.xyz_opt, self.measurements, native=native)
        self.optimal = r["outcome"] in (0, 2)
        if r["outcome"] in (1, 2):
            self.opt_success += 1
            self.xyz_opt = r["xyz"].copy()
        elif r["outcome"] in (3, 4):
            self.opt_failed += 1


class TrackerGT:
    def __init__(self, cam_l, cam_r, cfg, visible_min=100, max_gap=2, threads=1, native=False):
        self.cam_l, self.cam_r, self.cfg, self.threads, self.native = cam_l, cam_r, cfg, threads, native
        self.P_l, self.P_r = np.asarray(cam_l.P, np.float64).reshape(3, 4), np.asarray(cam_r.P, np.float64).reshape(3, 4)
        self.visible_min, self.max_gap = visible_min, max_gap
        self.points = []            # detection points: dict(T_l2w, landmarks)
        self.visible = []           # m_vecVisibleLandmarks
        self.T_w2l_last = np.eye(4)
        self.frame = self.visible_last = self.detections = self.gap = self.next_uid = 0
        self.tracks = (0, 0, 0)

    def active(self):
        return [lm for d in self.points for lm in d["landmarks"]]

    def process(self, L, R, T_last_to_now, rotation_norm=0.0):
        t = T_last_to_now[:3, 3]
        t_norm = float(np.sqrt(t[0] * t[0] + t[1] * t[1] + t[2] * t[2]))
        T_w2l = iso_mul(T_last_to_now, self.T_w2l_last)
        T_l2w = iso_inv(T_w2l)
        scaling = min(1.0 + (10.0 * rotation_norm + 0.5 * t_norm), 5.0)
        for lm in self.visible:
            lm.visible = False
        self.visible = []
        self._track_manual(L, R, T_w2l, T_l2w, scaling)
        self.visible_last = len(self.visible)
        for lm in self.active():
            lm.optimize()
        if self.visible_min > self.visible_last or self.max_gap < self.gap:
            self.visible_last = self._add_new(L, R, T_w2l, T_l2w)
            self.gap = 0
            self.detections += 1
        else:
            self.gap += 1
        self.T_w2l_last = T_w2l
        self.frame += 1

    def _track_manual(self, L, R, T_w2l, T_l2w, scaling):
        P_w2l, P_w2r = proj_mul(self.P_l, T_w2l), proj_mul(self.P_r, T_w2l)
        cand, tdet = [], []
        for d in self.points:
            for lm in d["landmarks"]:
                if 0 < lm.opt_failed:
                    lm.visible = lm.optimal = False
                elif 0 < lm.opt_success and not lm.optimal:
                    lm.visible = False
                else:
                    cand.append(lm)
                    tdet.append(d["T_l2w"])
        s1 = s2 = s3 = 0
        if cand:
            r = co.track_landmarks(self.cfg, L, R, T_w2l, np.array([lm.xyz_opt for lm in cand]), np.array([lm.last_desc_l for lm in cand]),
                                   np.array([lm.last_desc_r for lm in cand]), np.array([lm.last_disp for lm in cand], np.float32),
                                   np.array([lm.size for lm in cand], np.float32), scaling, uv_reference_left=np.array([lm.uv_ref for lm in cand]),
                                   desc_reference_left=np.array([lm.ref_desc_l for lm in cand]), T_left_to_world_at_detection=np.array(tdet),
                                   n_threads=self.threads, native=self.native)
            for i, lm in enumerate(cand):
                if r["stage"][i] > 0:
                    lm.visible, lm.failed = True, 0
                    lm.add_measurement(r["uv_l"][i], r["uv_r"][i], r["desc_l"][i], r["desc_r"][i], r["xyz"][i], P_w2l, P_w2r)
                    self.visible.append(lm)
                    if r["stage"][i] <= 2:
                        s1 += 1
                    elif r["stage"][i] <= 4:
                        s2 += 1
                    else:
                        s3 += 1
                elif r["status"][i] != ST_EPI_NO_TRANSLATION:
                    lm.failed += 1
                    lm.visible = False
        self.tracks = (s1, s2, s3)
        for d in self.points:
            d["landmarks"] = [lm for lm in d["landmarks"] if lm.failed < MAX_FAILED]
        self.points = [d for d in self.points if d["landmarks"]]

    def _mask_centres(self, T_w2l):
        c = []
        for lm in self.active():
            if lm.visible:
                c.append(lm.last_uv_l)
            else:
                p = iso_apply(T_w2l, lm.xyz_opt)
                P = self.P_l
                w = P[2, 0] * p[0] + P[2, 1] * p[1] + P[2, 2] * p[2] + P[2, 3]
                c.append((np.float32((P[0, 0] * p[0] + P[0, 1] * p[1] + P[0, 2] * p[2] + P[0, 3]) / w),
                          np.float32((P[1, 0] * p[0] + P[1, 1] * p[1] + P[1, 2] * p[2] + P[1, 3]) / w)))
        return np.asarray(c, np.float32).reshape(-1, 2)

    def _add_new(self, L, R, T_w2l, T_l2w):
        P_w2l, P_w2r = proj_mul(self.P_l, T_w2l), proj_mul(self.P_r, T_w2l)
        centres = self._mask_centres(T_w2l)
        ok = np.isfinite(centres).all(axis=1) & (np.abs(centres) < 1.0e6).all(axis=1) if len(centres) else np.zeros(0, bool)
        m = o.mask_active_landmarks(L.shape[1], L.shape[0], centres[ok])[None] if len(centres) else None
        d = co.frame(co.stereo_frames(self.cfg, L, R, masks=m, native=self.native), 0)
        new = []
        for u in range(len(d["status"])):
            if d["status"][u] != 0:
                continue
            lm = Landmark(self.next_uid, d["desc_l"][u], d["desc_r"][u], self.cfg.keypoint_size, d["uv_l"][u], d["uv_r"][u], d["xyz"][u], T_l2w, P_w2l, P_w2r)
            lm.optimal = True
            new.append(lm)
            self.next_uid += 1
        if not new:
            return 0
        self.points.append(dict(T_l2w=T_l2w.copy(), landmarks=new))
        return len(new)


# ------------------------------------------------------------------------------------------------- the stereo-only tracker
SV_CANDIDATE, SV_LEAVES = 1, 2                                   # flags: bIsOptimal | leaves in trackEpipolar
ROUTE_POSE, ROUTE_EPIPOLAR, ROUTE_REGIONAL, ROUTE_REGIONAL_NO_TRANSLATION, ROUTE_DROPPED = 1, 2, 3, 4, 5
POSIT_OK = 0
SV_SOURCES = ("posit", "posit-damped", "prior")
TRACK_KEYS = ("status", "stage", "uv_l", "uv_r", "xyz", "desc_l", "desc_r")


def translation_moved(T, T_det):
    """trackEpipolar :800: has the camera moved since the detection?  The translation column of T * T_det (Isometry3d product,
    the sum starting at 0.0), then 0 < its squared norm summed x, y, z."""
    t = []
    for r in range(3):
        s = 0.0
        for k in range(3):
            s = s + float(T[r, k]) * float(T_det[k, 3])
        t.append(s + float(T[r, 3]))
    return 0.0 < (t[0] * t[0] + t[1] * t[1]) + t[2] * t[2]


def _projections(cfg):
    return np.array(cfg.P_left[:], np.float64).reshape(3, 4), np.array(cfg.P_right[:], np.float64).reshape(3, 4)


def sv_frame(cfg, L, R, landmarks, flags, T_est, T_damped, T_last, t_imu, scaling, threads=1, native=False):
    """One frame of the stereo-only tracker, what StereoFrontend.track_frame_stereo_only returns, from the C restatement:
    getPoseStereoPosit (stages 1-2 on the candidates around the prior, the pose solve on their hits in candidate order) around
    T_est, again around T_damped if that solve fails, the pose T_damped if both fail (CTrackerSV.cpp:268-313); then trackEpipolar's
    split of every other landmark: the pose hits of an accepted solve are seen, a leaving landmark is dropped, the rest goes to
    stage 3 where the camera moved since its detection, else -- and where stage 3 finds no translation (:1804) -- to the regional
    stage 2.  landmarks: dict(xyz_w, last_desc_l, last_desc_r, last_disp, uv_ref, ref_desc_l, T_det) over all n landmarks."""
    P_l, P_r = _projections(cfg)
    flags = np.asarray(flags, np.uint8)
    n = len(flags)
    xyz_w = np.asarray(landmarks["xyz_w"], np.float64).reshape(n, 3)
    T_det = np.asarray(landmarks["T_det"], np.float64).reshape(n, 4, 4)

    def zeros():
        return dict(status=np.zeros(n, np.uint8), stage=np.zeros(n, np.uint8), uv_l=np.zeros((n, 2), np.float32), uv_r=np.zeros((n, 2), np.float32),
                    xyz=np.zeros((n, 3), np.float64), desc_l=np.zeros((n, 32), np.uint8), desc_r=np.zeros((n, 32), np.uint8))

    def track(idx, T, stages):
        idx = np.asarray(idx, np.int64)
        ref = dict(uv_reference_left=np.asarray(landmarks["uv_ref"])[idx], desc_reference_left=np.asarray(landmarks["ref_desc_l"])[idx],
                   T_left_to_world_at_detection=T_det[idx]) if stages & 4 else {}
        return co.track_landmarks(cfg, L, R, T, xyz_w[idx], np.asarray(landmarks["last_desc_l"])[idx], np.asarray(landmarks["last_desc_r"])[idx],
                                  np.asarray(landmarks["last_disp"], np.float32)[idx], cfg.keypoint_size, scaling, stages=stages, n_threads=threads,
                                  native=native, **ref)

    pose, epi = zeros(), zeros()
    cand = [i for i in range(n) if flags[i] & SV_CANDIDATE]
    attempts, measurements, accepted = [], [], None
    for a, T_prior in enumerate((T_est, T_damped)):
        r = track(cand, T_prior, 3)
        hits = [j for j in range(len(cand)) if r["stage"][j] > 0]
        measurements.append(len(hits))
        attempts.append(co.solve_stereo_posit(P_l, P_r, xyz_w[[cand[j] for j in hits]].reshape(-1, 3), r["uv_l"][hits], r["uv_r"][hits], T_prior,
                                              T_last, t_imu, native=native))
        for j, i in enumerate(cand):
            for k in TRACK_KEYS:
                pose[k][i] = r[k][j]
        if attempts[-1]["outcome"] == POSIT_OK:
            accepted = a
            break
    T = attempts[accepted]["T"].copy() if accepted is not None else np.asarray(T_damped, np.float64).copy()
    route = np.zeros(n, np.uint8)
    for i in range(n):
        if accepted is not None and pose["stage"][i] > 0:
            route[i] = ROUTE_POSE
        elif flags[i] & SV_LEAVES:
            route[i] = ROUTE_DROPPED
        else:
            route[i] = ROUTE_EPIPOLAR if translation_moved(T, T_det[i]) else ROUTE_REGIONAL
    for idx, stages in (([i for i in range(n) if route[i] == ROUTE_EPIPOLAR], 4), (None, 2)):
        if idx is None:   # the regional search: the unmoved landmarks and the stage-3 items without translation
            idx = [i for i in range(n) if route[i] in (ROUTE_REGIONAL, ROUTE_REGIONAL_NO_TRANSLATION)]
        if not idx:
            continue
        r = track(idx, T, stages)
        for j, i in enumerate(idx):
            for k in TRACK_KEYS:
                epi[k][i] = r[k][j]
            if stages == 4 and r["status"][j] == ST_EPI_NO_TRANSLATION:
                route[i] = ROUTE_REGIONAL_NO_TRANSLATION
    source = SV_SOURCES[2 if accepted is None else accepted]
    return dict(T=T, source=source, attempts=attempts, measurements=measurements, route=route, pose_stage=pose, epipolar_stage=epi)


def rodrigues(M):
    """cv::Rodrigues of the rotation of M (the motion-scaling term, CTrackerSV.cpp:243-254): axis * angle from the trace and the
    skew part; zero for the identity."""
    import math
    c = min(1.0, max(-1.0, ((float(M[0, 0]) + float(M[1, 1]) + float(M[2, 2])) - 1.0) / 2.0))
    angle = math.acos(c)
    rx, ry, rz = float(M[2, 1]) - float(M[1, 2]), float(M[0, 2]) - float(M[2, 0]), float(M[1, 0]) - float(M[0, 1])
    s2 = math.sqrt(rx * rx + ry * ry + rz * rz)
    if s2 < 1e-12:
        return (0.0, 0.0, 0.0)
    k = angle / s2
    return (k * rx, k * ry, k * rz)


def _norm3(v):
    import math
    return math.sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])


class TrackerSV(TrackerGT):
    """CTrackerSV::process without any given pose: the pose of each frame comes from the stereo solve on the landmarks
    tracked around a constant-velocity prior (sv_frame), and the landmark bookkeeping of getPoseStereoPosit / trackEpipolar
    follows.  Re-detection and the landmark model are TrackerGT's.  Per frame it leaves: source, tracks (S1, S2, S3, S22),
    visible (in measurement order), visible_last, instability, posit_last (size of the last accepted solve's problem),
    T_w2l_last and the active landmarks."""

    def __init__(self, cam_l, cam_r, cfg, visible_min=100, max_gap=2, optimize_every=10, threads=1, native=False):
        super().__init__(cam_l, cam_r, cfg, visible_min=visible_min, max_gap=max_gap, threads=threads, native=native)
        self.optimize_every = optimize_every
        self.T_motion = np.eye(4)          # m_matTransformationLEFTLASTtoLEFTNOW
        self.instability = self.posit_last = 0
        self.source, self.tracks, self.last = "", (0, 0, 0, 0), None

    def process(self, L, R):
        # the priors (:243-254): the last motion again, and its rotation alone
        M = self.T_motion
        M_rot = M.copy()
        M_rot[:3, 3] = 0.0
        t_motion = np.array([M[0, 3], M[1, 3], M[2, 3]])
        T_est, T_damped = iso_mul(M, self.T_w2l_last), iso_mul(M_rot, self.T_w2l_last)
        scaling = min(1.0 + (10.0 * _norm3(rodrigues(M)) + 0.5 * _norm3(t_motion)), 5.0)
        for lm in self.visible:   # resetVisibilityActiveLandmarks :257
            lm.visible = False
        self.visible = []
        T = self._track_frame(L, R, T_est, T_damped, t_motion, scaling)
        if self.source == "posit":
            self.instability = max(0, self.instability - 1)
        elif self.source == "prior" and self.instability < 20:
            self.instability += 5
        # a sudden loss of more than three quarters of the visible landmarks :333-349
        n_vis = len(self.visible)
        if 0 < self.visible_last and 0.75 < float(self.visible_last - n_vis) / float(self.visible_last) and self.instability < 20:
            self.instability += 5
        self.visible_last = n_vis
        if self.frame % self.optimize_every == 0:   # :362-365
            for lm in self.active():
                lm.optimize_exact(self.native)
        if self.visible_min > self.visible_last or self.max_gap < self.gap:   # :468-473
            self.visible_last = self._add_new(L, R, T, iso_inv(T))
            self.gap = 0
            self.detections += 1
        else:
            self.gap += 1
        self.frame += 1
        self.T_motion = iso_mul(T, iso_inv(self.T_w2l_last))   # :547-548
        self.T_w2l_last = T

    def _track_frame(self, L, R, T_est, T_damped, t_motion, scaling):
        lms, dets = [], []
        for d in self.points:
            for lm in d["landmarks"]:
                lms.append(lm)
                dets.append(d["T_l2w"])
        n = len(lms)
        flags = np.zeros(n, np.uint8)
        for i, lm in enumerate(lms):
            leaves = 0 < lm.opt_failed or (0 < lm.opt_success and not lm.optimal)   # :808-825
            flags[i] = (SV_CANDIDATE if lm.optimal else 0) | (SV_LEAVES if leaves else 0)
        st = dict(xyz_w=np.array([lm.xyz_opt for lm in lms]).reshape(n, 3), last_desc_l=np.array([lm.last_desc_l for lm in lms], np.uint8).reshape(n, 32),
                  last_desc_r=np.array([lm.last_desc_r for lm in lms], np.uint8).reshape(n, 32),
                  last_disp=np.array([lm.last_disp for lm in lms], np.float32), uv_ref=np.array([lm.uv_ref for lm in lms]).reshape(n, 2),
                  ref_desc_l=np.array([lm.ref_desc_l for lm in lms], np.uint8).reshape(n, 32), T_det=np.array(dets).reshape(n, 4, 4))
        r = sv_frame(self.cfg, L, R, st, flags, T_est, T_damped, self.T_w2l_last, t_motion, scaling, threads=self.threads, native=self.native)
        self.last = r
        self.source = r["source"]
        T = r["T"]
        P_w2l, P_w2r = proj_mul(self.P_l, T), proj_mul(self.P_r, T)

        def measure(lm, res, i):
            lm.visible, lm.failed = True, 0
            lm.add_measurement(res["uv_l"][i], res["uv_r"][i], res["desc_l"][i], res["desc_r"][i], res["xyz"][i], P_w2l, P_w2r)
            self.visible.append(lm)

        # getPoseStereoPosit: the counters count the hits of the last solve even when it failed; only an accepted solve's hits
        # are measured, in candidate order, and become the last problem
        pose = r["pose_stage"]
        s1 = sum(1 for i in range(n) if 0 < pose["stage"][i] <= 2)
        s2 = sum(1 for i in range(n) if pose["stage"][i] > 2)
        if self.source != "prior":
            hits = [i for i in range(n) if pose["stage"][i] > 0]
            for i in hits:
                measure(lms[i], pose, i)
            self.posit_last = len(hits)
        # trackEpipolar: the leaving ones are not visible; stage 3, then the regional stage 2 (unmoved, then re-routed), each in
        # landmark order; a miss counts as a failed tracking
        epi, route = r["epipolar_stage"], r["route"]
        for i in range(n):
            if flags[i] & SV_LEAVES:
                lms[i].visible = False
        counts = {}
        for rt in (ROUTE_EPIPOLAR, ROUTE_REGIONAL, ROUTE_REGIONAL_NO_TRANSLATION):
            counts[rt] = 0
            for i in range(n):
                if route[i] != rt:
                    continue
                if epi["stage"][i] > 0:
                    measure(lms[i], epi, i)
                    counts[rt] += 1
                else:
                    lms[i].failed += 1
                    lms[i].visible = False
        self.tracks = (s1, s2, counts[ROUTE_EPIPOLAR], counts[ROUTE_REGIONAL] + counts[ROUTE_REGIONAL_NO_TRANSLATION])
        # activity :1291-1312: the leaving ones and those with MAX_FAILED failed trackings go
        gone = {id(lms[i]) for i in range(n) if flags[i] & SV_LEAVES or lms[i].failed >= MAX_FAILED}
        for d in self.points:
            d["landmarks"] = [lm for lm in d["landmarks"] if id(lm) not in gone]
        self.points = [d for d in self.points if d["landmarks"]]
        return T
